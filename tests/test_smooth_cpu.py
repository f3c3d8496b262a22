"""CPU tests of the fixed-interval smoother: the NumPy recursion against a solver-independent MAP certificate, the storage query
of optistate_kf_smooth_storage_bytes, and the descriptor refusals of optistate_kf_smooth (all before any CUDA call)."""
import ctypes

import numpy as np
import pytest

from oracle import cases
from tests import rts_oracle as ro
from tests.test_abi_cpu import _valid_desc, lib  # noqa: F401 - the fixture


@pytest.mark.parametrize("name", ["cfg1_default_seed0", "stress_qrpkl_seed3_10k"])
def test_rts_recursion_equals_map_certificate(name):
    stream, kw, _ = cases.build(name)
    s = {k: v[:40] for k, v in stream.items()}
    fw = ro.forward(s, kw["x0"], kw["P0"], kw["Q"], kw["R"])
    xs, Ps = ro.rts(fw["x"], fw["x_model"], fw["P"], kw["Q"])
    P0 = kw["Q"] if kw["P0"] is None else kw["P0"]
    mean, cov = ro.map_certificate(kw["x0"], P0, kw["Q"], kw["R"], fw["x"], fw["x_model"], fw["z"])
    scale = np.abs(mean).max(axis=0)
    scale = np.where(scale > 0, scale, 1.0)
    assert (np.abs(xs - mean).max(axis=0) / scale).max() <= 1e-10
    assert np.abs(Ps - cov).max() <= 1e-10 * np.abs(cov).max()
    # smoothing uses the later measurements: it moves the estimate, and never widens the marginal variances
    assert np.abs(xs[:-1] - fw["x"][:-1]).max() > 0
    assert (np.einsum("tii->ti", Ps) <= np.einsum("tii->ti", fw["P"]) * (1 + 1e-12)).all()


class SmoothDesc(ctypes.Structure):
    """ctypes mirror of OptiKfSmoothDesc."""
    _fields_ = [("struct_size", ctypes.c_uint32), ("abi_version", ctypes.c_uint32), ("filter", ctypes.c_void_p),
                ("x_smooth", ctypes.c_void_p), ("var_smooth", ctypes.c_void_p), ("storage", ctypes.c_void_p),
                ("storage_bytes", ctypes.c_size_t)]


def _storage(lib, d):  # noqa: F811
    n = ctypes.c_size_t(123)
    rc = lib.optistate_kf_smooth_storage_bytes(ctypes.byref(d), ctypes.byref(n))
    return rc, n.value


def test_storage_holds_packed_covariance_and_missing_estimates(lib):  # noqa: F811
    d = _valid_desc(lib)
    d.n_traj, d.n_streams, d.n_steps = 1000, 100, 37
    up = lambda b: (b + 255) // 256 * 256  # noqa: E731
    for dtype, esz in ((0, 8), (1, 4)):
        d.dtype = dtype
        tn = d.n_steps * d.n_traj
        d.x_steps = d.x_model_steps = None
        assert _storage(lib, d) == (0, up(tn * 30 * esz) + 2 * up(tn * 12 * esz))
        d.x_steps = ctypes.c_void_p(0x1000)  # the smoother reads the caller's x_steps instead
        assert _storage(lib, d) == (0, up(tn * 30 * esz) + up(tn * 12 * esz))
        d.x_model_steps = ctypes.c_void_p(0x2000)
        assert _storage(lib, d) == (0, up(tn * 30 * esz))


def test_refusals_return_their_codes(lib):  # noqa: F811
    f = _valid_desc(lib)
    s = SmoothDesc(ctypes.sizeof(SmoothDesc), lib.optistate_kf_abi_version(), ctypes.addressof(f), 0x1000, None, 0x1000, 1 << 30)

    def rc(desc=s):
        return lib.optistate_kf_smooth(ctypes.byref(desc), None)

    assert lib.optistate_kf_smooth(None, None) == -1
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
    for field, value in (("algo", 1), ("q_kind", 3), ("r_kind", 4), ("p0_kind", 3), ("cov_model", 1), ("flags", 2)):
        f2 = _valid_desc(lib)
        setattr(f2, field, value)
        if field == "p0_kind":
            f2.P0 = ctypes.c_void_p(0x1000)
        if field == "cov_model":
            f2.body_ref = ctypes.c_void_p(0x1000)
        s2 = SmoothDesc.from_buffer_copy(s)
        s2.filter = ctypes.addressof(f2)
        assert rc(s2) == -5, field
        assert _storage(lib, f2)[0] == -5, field
    f3 = _valid_desc(lib)  # a dense P0 that the caller vouches for as decoupled is taken
    f3.p0_kind, f3.P0, f3.flags, f3.algo = 3, ctypes.c_void_p(0x1000), 1, 2
    assert _storage(lib, f3)[0] == 0
