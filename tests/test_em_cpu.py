"""CPU tests of the EM E-step: the textbook oracle against the dense certificate, the EM theorem on a frozen linearisation, and the
storage query and descriptor refusals of optistate_kf_noise_em_stats (all before any CUDA call)."""
import ctypes

import numpy as np
import pytest

from oracle import cases
from tests import em_oracle as eo
from tests.test_abi_cpu import _valid_desc, lib  # noqa: F401 - the fixture
from tests.test_smooth_cpu import _storage as _smooth_storage


def _kw(name, T):
    stream, kw, _ = cases.build(name)
    s = {k: v[:T] for k, v in stream.items()}
    P0 = kw["Q"] if kw["P0"] is None else kw["P0"]
    return s, kw, P0


@pytest.mark.parametrize("name", ["cfg1_default_seed0", "stress_qrpkl_seed3_10k"])
def test_textbook_estep_equals_dense_certificate(name):
    s, kw, P0 = _kw(name, 40)
    ch = eo.forward(s, kw["x0"], P0, kw["Q"], kw["R"])
    Sw, Sv, ll = eo.estep_textbook(ch, kw["Q"], kw["R"])
    Sw2, Sv2, ll2 = eo.estep_dense(ch, kw["Q"], kw["R"])
    assert np.abs(Sw - Sw2).max() <= 1e-10 * np.abs(Sw2).max()
    assert (np.abs(Sw - Sw2) <= 1e-10 * np.abs(Sw2)).all()
    assert (np.abs(Sv - Sv2) <= 1e-10 * np.abs(Sv2)).all()
    assert abs(ll - ll2) <= 1e-10 * abs(ll2)


def test_em_never_decreases_with_frozen_linearisation():
    """With F and the offsets of the affine model fixed from one forward pass, EM is exact EM: the likelihood never falls."""
    s, kw, P0 = _kw("cfg1_default_seed0", 60)
    q, r = np.diag(kw["Q"]) * 10.0, np.diag(kw["R"]) * 0.1
    ch0 = eo.forward(s, kw["x0"], np.diag(q), np.diag(q), np.diag(r))
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


class EmDesc(ctypes.Structure):
    """ctypes mirror of OptiKfNoiseEmDesc."""
    _fields_ = [("struct_size", ctypes.c_uint32), ("abi_version", ctypes.c_uint32), ("filter", ctypes.c_void_p),
                ("stats", ctypes.c_void_p), ("x_smooth", ctypes.c_void_p), ("var_smooth", ctypes.c_void_p),
                ("storage", ctypes.c_void_p), ("storage_bytes", ctypes.c_size_t)]


def _storage(lib, d):  # noqa: F811
    n = ctypes.c_size_t(123)
    rc = lib.optistate_kf_noise_em_storage_bytes(ctypes.byref(d), ctypes.byref(n))
    return rc, n.value


def test_storage_is_the_smoothers_plus_measurements(lib):  # noqa: F811
    d = _valid_desc(lib)
    d.n_traj, d.n_streams, d.n_steps = 1000, 100, 37
    up = lambda b: (b + 255) // 256 * 256  # noqa: E731
    for dtype, esz in ((0, 8), (1, 4)):
        d.dtype = dtype
        d.x_steps = d.x_model_steps = None
        rc, smooth = _smooth_storage(lib, d)
        assert rc == 0
        assert d.phases == 7  # the filter forms z: the E-step forms it once more into the storage
        assert _storage(lib, d) == (0, smooth + up(37 * 10 * 100 * esz))
        d.phases, d.z_in = 6, ctypes.c_void_p(0x3000)  # caller-supplied z is read where it is
        assert _storage(lib, d) == (0, smooth)
        d.phases, d.z_in = 7, None


def test_refusals_return_their_codes(lib):  # noqa: F811
    f = _valid_desc(lib)
    s = EmDesc(ctypes.sizeof(EmDesc), lib.optistate_kf_abi_version(), ctypes.addressof(f), 0x1000, None, None, 0x1000, 1 << 30)

    def rc(desc=s):
        return lib.optistate_kf_noise_em_stats(ctypes.byref(desc), None)

    assert lib.optistate_kf_noise_em_stats(None, None) == -1
    for field, value, code in (("struct_size", ctypes.sizeof(EmDesc) - 8, -2), ("abi_version", s.abi_version + 1, -2),
                               ("filter", None, -1), ("stats", None, -1), ("storage_bytes", 100, -4)):
        bad = EmDesc.from_buffer_copy(s)
        setattr(bad, field, value)
        assert rc(bad) == code, field
    for field, value in (("algo", 1), ("q_kind", 3), ("r_kind", 4), ("p0_kind", 3), ("cov_model", 1), ("flags", 2)):
        f2 = _valid_desc(lib)
        setattr(f2, field, value)
        if field == "p0_kind":
            f2.P0 = ctypes.c_void_p(0x1000)
        if field == "cov_model":
            f2.body_ref = ctypes.c_void_p(0x1000)
        s2 = EmDesc.from_buffer_copy(s)
        s2.filter = ctypes.addressof(f2)
        assert rc(s2) == -5, field
        assert _storage(lib, f2)[0] == -5, field
    f3 = _valid_desc(lib)  # a dense P0 that the caller vouches for as decoupled is taken
    f3.p0_kind, f3.P0, f3.flags, f3.algo = 3, ctypes.c_void_p(0x1000), 1, 2
    assert _storage(lib, f3)[0] == 0
