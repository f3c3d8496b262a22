"""CPU tests of the four backward entries' storage queries (pure host code): over a grid of filter descriptors, each E-step
accepts exactly what its smoother accepts, with the same return codes (include/optistate_kf.h), and where they accept, the
storage is P+ [T][np][N], the missing x+ / x- [T][12][N], and for the E-step the formed z [T][10][S], each padded to 256 B."""
import ctypes
import itertools

from tests.test_abi_cpu import _valid_desc, lib  # noqa: F401 - the fixture

N, S = 1000, 100
FAKE = ctypes.c_void_p(0x1000)  # never dereferenced: the queries only validate


def _up(b):
    return (b + 255) // 256 * 256


def _query(fn, d):
    n = ctypes.c_size_t(123)
    return fn(ctypes.byref(d), ctypes.byref(n)), n.value


def test_estep_queries_match_their_smoothers_over_a_descriptor_grid(lib):  # noqa: F811
    pairs = ((lib.optistate_kf_smooth_storage_bytes, lib.optistate_kf_noise_em_storage_bytes, 30),
             (lib.optistate_kf_smooth_full_storage_bytes, lib.optistate_kf_noise_em_full_storage_bytes, 78))
    accepted = [0, 0]
    refused = [set(), set()]
    d = _valid_desc(lib)
    d.n_traj, d.n_streams = N, S
    grid = itertools.product((0, 1), (0, 1, 2), (0, 1), (0, 1, 2, 3), (0, 1, 2, 3, 4), (1, 2, 3, 4), (1, 2, 3, 4), (True, False),
                             (False, True), (False, True), (False, True), (0, 37))
    for dtype, algo, cov, flags, p0k, qk, rk, formed, xs, xm, ref, T in grid:
        d.dtype, d.algo, d.cov_model, d.flags, d.n_steps = dtype, algo, cov, flags, T
        d.p0_kind, d.q_kind, d.r_kind = p0k, qk, rk
        d.P0 = FAKE if p0k else None
        d.phases, d.z_in = (7, None) if formed else (6, FAKE)
        d.x_steps = FAKE if xs else None
        d.x_model_steps = FAKE if xm else None
        d.body_ref = FAKE if ref else None
        esz = 8 if dtype == 0 else 4
        point = (dtype, algo, cov, flags, p0k, qk, rk, formed, xs, xm, ref, T)
        for k, (smooth_q, em_q, np_) in enumerate(pairs):
            rc, smooth = _query(smooth_q, d)
            rc_em, em = _query(em_q, d)
            assert rc_em == rc, (k, point)
            if rc != 0:
                refused[k].add(rc)
                continue
            accepted[k] += 1
            x = _up(T * N * 12 * esz)
            assert smooth == _up(T * N * np_ * esz) + (0 if xs else x) + (0 if xm else x), (k, point)
            assert em == smooth + (_up(T * 10 * S * esz) if formed else 0), (k, point)
    # the grid reaches acceptance and the refusals of both families
    assert min(accepted) > 0, accepted
    assert refused[0] >= {-1, -5} and refused[1] >= {-1, -5}, refused
