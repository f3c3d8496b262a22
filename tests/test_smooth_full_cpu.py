"""CPU tests of the full-covariance smoother: the NumPy recursion of tests/rts_full_oracle.py against the dense MAP certificate for
both covariance models, and the storage query and descriptor checks of optistate_kf_smooth_full (all before any CUDA call)."""
import ctypes

import numpy as np
import pytest

from oracle import cases
from optistate_b200.synth import make_stream
from tests import rts_full_oracle as rf
from tests.test_abi_cpu import _valid_desc, lib  # noqa: F401 - the fixture
from tests.test_smooth_cpu import SmoothDesc


def _case(name, T):
    """(stream, kw, model) on make_stream(5, T) with body_ref = truth: the next_mpc_cov_seed5 set-up and its variants."""
    s = make_stream(5, T)
    s["body_ref"] = s["truth"].copy()
    kw = dict(x0=cases.START.copy(), P0=None, Q=cases.Q_DEFAULT.copy(), R=cases.R_DEFAULT.copy())
    if name == "predict_coupled_p0":
        rng = np.random.default_rng(77)
        A = rng.standard_normal((12, 12))
        kw["P0"] = 0.02 * (A @ A.T / 12 + 0.5 * np.eye(12))
        return s, kw, "predict"
    if name == "mpc_default":
        return s, kw, "mpc"
    kw["Q"], kw["R"] = cases.q_r_pkl()
    return s, kw, "mpc" if name == "mpc_qrpkl" else "predict"


@pytest.mark.parametrize("name", ["predict_coupled_p0", "mpc_default", "predict_qrpkl"])
def test_full_rts_equals_map_certificate(name):
    s, kw, model = _case(name, 40)
    fw = rf.forward(s, kw["x0"], kw["P0"], kw["Q"], kw["R"], model)
    xs, Ps = rf.rts(fw["x"], fw["x_model"], fw["P"], kw["Q"], fw["F"])
    P0 = kw["Q"] if kw["P0"] is None else kw["P0"]
    mean, cov = rf.map_certificate(kw["x0"], P0, kw["Q"], kw["R"], fw["x"], fw["x_model"], fw["z"], fw["F"])
    ex, ev = rf.rel_errors(xs, Ps, mean, np.einsum("tii->ti", cov))
    assert ex <= 1e-10 and ev <= 1e-10, (ex, ev)
    assert np.abs(xs[:-1] - fw["x"][:-1]).max() > 0
    assert (np.einsum("tii->ti", Ps) <= np.einsum("tii->ti", fw["P"]) * (1 + 1e-12)).all()
    # the transitions rebuilt from the run alone (what the backward kernel does) are the ones the filter used
    F = rf.transitions(fw["x"], model, s["body_ref"], kw["x0"])
    assert np.array_equal(F, fw["F"])
    if model == "mpc":  # predict_mpc couples the groups: the decoupled smoother could not take this P
        assert np.abs(fw["P"][:, 0, 3]).max() > 0


def test_qrpkl_mpc_solve_equals_cholesky():
    """Q_R.pkl noise under predict_mpc: cond(P-) is ~5e7 at the median and reaches ~1e8, so the dense certificate's own inverse is
    the weak part (1e-6 from the recursion) and it is not used here.  Two FP64 solvers of the recursion agree instead: LU
    (np.linalg.solve) against Cholesky, 2,000 steps.  Measured: x 5.4e-9 (the body rate w_z; 6.8e-9 at 10,000 steps), var 1.4e-9,
    both relative to each state's largest value (DESIGN.md section 0.2); the bounds leave a factor of ~4."""
    s, kw, model = _case("mpc_qrpkl", 2000)
    fw = rf.forward(s, kw["x0"], kw["P0"], kw["Q"], kw["R"], model)
    xa, Pa = rf.rts(fw["x"], fw["x_model"], fw["P"], kw["Q"], fw["F"], "solve")
    xb, Pb = rf.rts(fw["x"], fw["x_model"], fw["P"], kw["Q"], fw["F"], "cholesky")
    ex, ev = rf.rel_errors(xa, Pa, xb, np.einsum("tii->ti", Pb))
    assert ex <= 2e-8 and ev <= 5e-9, (ex, ev)


def _storage(lib, d):  # noqa: F811
    n = ctypes.c_size_t(123)
    rc = lib.optistate_kf_smooth_full_storage_bytes(ctypes.byref(d), ctypes.byref(n))
    return rc, n.value


def test_storage_holds_full_covariance_and_missing_estimates(lib):  # noqa: F811
    d = _valid_desc(lib)
    d.n_traj, d.n_streams, d.n_steps = 1000, 100, 37
    up = lambda b: (b + 255) // 256 * 256  # noqa: E731
    for dtype, esz in ((0, 8), (1, 4)):
        d.dtype = dtype
        tn = d.n_steps * d.n_traj
        d.x_steps = d.x_model_steps = None
        assert _storage(lib, d) == (0, up(tn * 78 * esz) + 2 * up(tn * 12 * esz))
        d.x_steps = ctypes.c_void_p(0x1000)
        assert _storage(lib, d) == (0, up(tn * 78 * esz) + up(tn * 12 * esz))
        d.x_model_steps = ctypes.c_void_p(0x2000)
        assert _storage(lib, d) == (0, up(tn * 78 * esz))


def test_refusals_return_their_codes(lib):  # noqa: F811
    f = _valid_desc(lib)
    s = SmoothDesc(ctypes.sizeof(SmoothDesc), lib.optistate_kf_abi_version(), ctypes.addressof(f), 0x1000, None, 0x1000, 1 << 30)

    def rc(desc=s):
        return lib.optistate_kf_smooth_full(ctypes.byref(desc), None)

    assert lib.optistate_kf_smooth_full(None, None) == -1
    bad = SmoothDesc.from_buffer_copy(s)
    bad.struct_size -= 8
    assert rc(bad) == -2
    bad = SmoothDesc.from_buffer_copy(s)
    bad.abi_version += 1
    assert rc(bad) == -2
    bad = SmoothDesc.from_buffer_copy(s)
    bad.filter = None
    assert rc(bad) == -1
    bad = SmoothDesc.from_buffer_copy(s)
    bad.x_smooth = None
    assert rc(bad) == -1
    bad = SmoothDesc.from_buffer_copy(s)
    bad.storage_bytes = 100
    assert rc(bad) == -4
    # what the sequential filter cannot run
    for field, value in (("algo", 1), ("q_kind", 3), ("r_kind", 4)):
        f2 = _valid_desc(lib)
        setattr(f2, field, value)
        s2 = SmoothDesc.from_buffer_copy(s)
        s2.filter = ctypes.addressof(f2)
        assert rc(s2) == -5, field
        assert _storage(lib, f2)[0] == -5, field
    f2 = _valid_desc(lib)
    f2.dtype = 7
    assert _storage(lib, f2)[0] == -3
    assert lib.optistate_kf_smooth_full_storage_bytes(ctypes.byref(_valid_desc(lib)), None) == -1


def test_takes_what_the_decoupled_smoother_refuses(lib):  # noqa: F811
    """The predict_mpc model, the full-covariance flag and dense P0 kinds: refused by optistate_kf_smooth, taken here."""
    for field, value in (("p0_kind", 3), ("p0_kind", 4), ("cov_model", 1), ("flags", 2)):
        for algo in (0, 2):
            f2 = _valid_desc(lib)
            f2.algo = algo
            setattr(f2, field, value)
            if field == "p0_kind":
                f2.P0 = ctypes.c_void_p(0x1000)
            if field == "cov_model":
                f2.body_ref = ctypes.c_void_p(0x1000)
            n = ctypes.c_size_t(0)
            assert lib.optistate_kf_smooth_storage_bytes(ctypes.byref(f2), ctypes.byref(n)) == -5, field
            assert _storage(lib, f2)[0] == 0, (field, algo)
    f2 = _valid_desc(lib)  # the predict_mpc model still needs its reference angles
    f2.cov_model = 1
    assert _storage(lib, f2)[0] == -1
