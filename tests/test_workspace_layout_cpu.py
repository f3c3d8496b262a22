"""CPU tests of the scratch the streamed SEQUENTIAL path asks for: besides z and the per-stream status it holds the leg
moments of the mean model ([T][12][S]), formed by the pre-pass once per base stream - also when the caller supplies z."""
import ctypes

from tests.test_abi_cpu import _valid_desc, lib  # noqa: F401 - the fixture


def _query(lib, d):  # noqa: F811
    n = ctypes.c_size_t(123)
    assert lib.optistate_kf_workspace_bytes(ctypes.byref(d), ctypes.byref(n)) == 0
    return n.value


def test_workspace_holds_measurements_moments_and_status(lib):  # noqa: F811
    d = _valid_desc(lib)
    d.n_streams, d.n_traj = 256, 1024
    T, S = d.n_steps, d.n_streams
    for dtype, esz in ((0, 8), (1, 4)):
        d.dtype = dtype
        assert _query(lib, d) >= T * (10 + 12) * S * esz + 4 * S


def test_workspace_with_preformed_measurements_holds_the_moments(lib):  # noqa: F811
    d = _valid_desc(lib)
    d.n_streams, d.n_traj = 256, 1024
    d.phases = 2 | 4  # PREDICT | UPDATE on a caller-supplied z
    d.z_in = ctypes.c_void_p(0x1000)
    assert _query(lib, d) >= d.n_steps * 12 * d.n_streams * 8
    d.n_streams = 100  # no 32-stream tiles: the direct-load kernel forms the moments itself
    assert _query(lib, d) == 0
