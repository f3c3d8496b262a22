"""CPU tests of the E-step on the full covariance: the textbook E-step of tests/em_oracle.py, fed the chains of
tests/em_full_oracle.py, against the dense certificate under both covariance models; two solvers where the certificate is too
ill-conditioned; the EM theorem on a frozen predict_mpc linearisation; and the storage query and descriptor checks of
optistate_kf_noise_em_full_stats (all before any CUDA call)."""
import ctypes

import numpy as np
import pytest

from oracle import cases
from tests import em_full_oracle as ef
from tests import em_oracle as eo
from tests.test_abi_cpu import _valid_desc, lib  # noqa: F401 - the fixture
from tests.test_em_cpu import EmDesc
from tests.test_smooth_full_cpu import _case
from tests.test_smooth_full_cpu import _storage as _smooth_full_storage


def _setup(name, T):
    """(stream, kw, model, P0): predict with a coupled P0, mpc with default noise, mpc with a coupled P0, mpc with Q_R.pkl."""
    if name == "mpc_coupled_p0":
        s, kw, _ = _case("predict_coupled_p0", T)
        model = "mpc"
    else:
        s, kw, model = _case(name, T)
    P0 = kw["Q"] if kw["P0"] is None else kw["P0"]
    return s, kw, model, P0


@pytest.mark.parametrize("name", ["predict_coupled_p0", "mpc_default", "mpc_coupled_p0"])
def test_textbook_estep_equals_dense_certificate(name):
    s, kw, model, P0 = _setup(name, 40)
    ch = ef.forward(s, kw["x0"], P0, kw["Q"], kw["R"], model)
    if model == "mpc":  # the chain is dense: the decoupled E-step could not take it
        assert np.abs(ch["PP"][1:, 0, 3]).max() > 0
    Sw, Sv, ll = eo.estep_textbook(ch, kw["Q"], kw["R"])
    Sw2, Sv2, ll_prior = eo.estep_dense(ch, kw["Q"], kw["R"])
    ll2 = ef.loglik_dense(ch, kw["Q"], kw["R"])  # em_oracle's dense likelihood inverts the prior, which predict_mpc makes meaningless
    assert (np.abs(Sw - Sw2) <= 1e-10 * np.abs(Sw2)).all(), np.abs(Sw - Sw2) / np.abs(Sw2)
    assert (np.abs(Sv - Sv2) <= 1e-10 * np.abs(Sv2)).all(), np.abs(Sv - Sv2) / np.abs(Sv2)
    assert abs(ll - ll2) <= 1e-10 * abs(ll2)
    if model == "predict":  # there both dense likelihoods are well posed and agree
        assert abs(ll_prior - ll2) <= 1e-10 * abs(ll2)


def test_qrpkl_mpc_lu_equals_cholesky():
    """Q_R.pkl noise under predict_mpc: cond(P-) ~5e7 makes the dense certificate's inverse the weak part (DESIGN.md section 0.2),
    so two FP64 solvers of the textbook recursion are compared instead, 2,000 steps.  Observed: Sw 1.5e-9, Sv 1.0e-11, log-likelihood
    3.7e-12 (relative, worst row); the bounds leave a factor of 3 to 5."""
    s, kw, model, P0 = _setup("mpc_qrpkl", 2000)
    ch = ef.forward(s, kw["x0"], P0, kw["Q"], kw["R"], model)
    Sw, Sv, ll = eo.estep_textbook(ch, kw["Q"], kw["R"])
    Sw2, Sv2, ll2 = ef.estep_cholesky(ch, kw["Q"], kw["R"])
    ew, ev, el = (float((np.abs(a - b) / np.abs(b)).max()) for a, b in ((Sw, Sw2), (Sv, Sv2), (ll, ll2)))
    print(f"Q_R.pkl mpc, LU vs Cholesky: Sw {ew:.1e}, Sv {ev:.1e}, loglik {el:.1e}")
    assert ew <= 5e-9 and ev <= 5e-11 and el <= 2e-11


def test_em_never_decreases_with_frozen_mpc_linearisation():
    """With the predict_mpc F sequence and the affine model's offsets frozen from one forward pass, EM is exact EM."""
    s, kw, model, _ = _setup("mpc_default", 60)
    q, r = np.diag(kw["Q"]) * 10.0, np.diag(kw["R"]) * 0.1
    ch0 = ef.forward(s, kw["x0"], np.diag(q), np.diag(q), np.diag(r), model)
    Fs, c = ch0["Fs"], [ch0["xm"][k] - ch0["Fs"][k] @ ch0["Xp"][k] for k in range(60)]
    lls = []
    for _ in range(12):
        ch = eo.linear_forward(Fs, c, ch0["Xp"][0], np.diag(np.diag(kw["Q"]) * 10.0), np.diag(q), np.diag(r), ch0["z"])
        Sw, Sv, ll = eo.estep_textbook(ch, np.diag(q), np.diag(r))
        lls.append(ll)
        q, r = Sw / 60, Sv / 60
    d = np.diff(lls)
    assert (d >= -1e-9 * np.abs(lls[1:])).all(), lls
    assert lls[-1] > lls[0]


def _storage(lib, d):  # noqa: F811
    n = ctypes.c_size_t(123)
    rc = lib.optistate_kf_noise_em_full_storage_bytes(ctypes.byref(d), ctypes.byref(n))
    return rc, n.value


def test_storage_is_the_full_smoothers_plus_measurements(lib):  # noqa: F811
    d = _valid_desc(lib)
    d.n_traj, d.n_streams, d.n_steps = 1000, 100, 37
    up = lambda b: (b + 255) // 256 * 256  # noqa: E731
    for dtype, esz in ((0, 8), (1, 4)):
        d.dtype = dtype
        d.x_steps = d.x_model_steps = None
        rc, smooth = _smooth_full_storage(lib, d)
        assert rc == 0 and smooth == up(37 * 1000 * 78 * esz) + 2 * up(37 * 1000 * 12 * esz)
        assert _storage(lib, d) == (0, smooth + up(37 * 10 * 100 * esz))
        d.phases, d.z_in = 6, ctypes.c_void_p(0x3000)  # caller-supplied z is read where it is
        assert _storage(lib, d) == (0, smooth)
        d.phases, d.z_in = 7, None


def test_refusals_return_their_codes(lib):  # noqa: F811
    f = _valid_desc(lib)
    s = EmDesc(ctypes.sizeof(EmDesc), lib.optistate_kf_abi_version(), ctypes.addressof(f), 0x1000, None, None, 0x1000, 1 << 30)

    def rc(desc=s):
        return lib.optistate_kf_noise_em_full_stats(ctypes.byref(desc), None)

    assert lib.optistate_kf_noise_em_full_stats(None, None) == -1
    for field, value, code in (("struct_size", ctypes.sizeof(EmDesc) - 8, -2), ("abi_version", s.abi_version + 1, -2),
                               ("filter", None, -1), ("stats", None, -1), ("storage_bytes", 100, -4)):
        bad = EmDesc.from_buffer_copy(s)
        setattr(bad, field, value)
        assert rc(bad) == code, field
    for field, value in (("algo", 1), ("q_kind", 3), ("r_kind", 4)):  # JOINT, dense Q, dense R
        f2 = _valid_desc(lib)
        setattr(f2, field, value)
        s2 = EmDesc.from_buffer_copy(s)
        s2.filter = ctypes.addressof(f2)
        assert rc(s2) == -5, field
        assert _storage(lib, f2)[0] == -5, field
    assert lib.optistate_kf_noise_em_full_storage_bytes(ctypes.byref(_valid_desc(lib)), None) == -1


def test_takes_what_the_decoupled_estep_refuses(lib):  # noqa: F811
    """The predict_mpc model, the full-covariance flag and a dense coupled P0: refused by optistate_kf_noise_em_stats, taken here."""
    for field, value in (("cov_model", 1), ("flags", 2), ("p0_kind", 3), ("p0_kind", 4)):
        for algo in (0, 2):
            f2 = _valid_desc(lib)
            f2.algo = algo
            setattr(f2, field, value)
            if field == "p0_kind":
                f2.P0 = ctypes.c_void_p(0x1000)
            if field == "cov_model":
                f2.body_ref = ctypes.c_void_p(0x1000)
            n = ctypes.c_size_t(0)
            assert lib.optistate_kf_noise_em_storage_bytes(ctypes.byref(f2), ctypes.byref(n)) == -5, field
            assert _storage(lib, f2)[0] == 0, (field, algo)
    f2 = _valid_desc(lib)  # the predict_mpc model still needs its reference angles
    f2.cov_model = 1
    assert _storage(lib, f2)[0] == -1
