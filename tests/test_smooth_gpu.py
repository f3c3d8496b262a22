"""GPU tests of the fixed-interval smoother (kf_smooth): the CUDA backward kernel against the NumPy recursion of
tests/rts_oracle.py, the forward pass it runs against kf_batch, and its properties and refusals."""
import numpy as np
import pytest
import torch

from oracle import cases
from optistate_b200 import kf_batch, kf_smooth
from optistate_b200.synth import make_streams, monte_carlo_noise
from tests import rts_oracle as ro

pytestmark = pytest.mark.gpu


def _streams(S, T, seed0):
    return make_streams(range(seed0, seed0 + S), T)


def _args(st):
    return st["imu"], st["p"], st["dp"], st["contact"], st["f"]


def _errors(res, st, kw, n):
    """Largest per-state error of x_smooth (relative to the state's max) and of var_smooth (relative to its max) over n streams."""
    ex = ev = 0.0
    xs_all, vs_all = res.x_smooth.cpu().numpy().astype(np.float64), res.var_smooth.cpu().numpy().astype(np.float64)
    for j in range(n):
        s = {k: v[:, :, j] for k, v in st.items()}
        fw = ro.forward(s, kw["x0"], kw["P0"], kw["Q"], kw["R"])
        xs, Ps = ro.rts(fw["x"], fw["x_model"], fw["P"], kw["Q"])
        var = np.einsum("tii->ti", Ps)
        scale = np.abs(xs).max(axis=0)
        scale = np.where(scale > 0, scale, 1.0)
        ex = max(ex, float((np.abs(xs_all[:, :, j] - xs).max(axis=0) / scale).max()))
        ev = max(ev, float(np.abs(vs_all[:, :, j] - var).max() / np.abs(var).max()))
    return ex, ev


@pytest.mark.parametrize("name", ["default_seed11_10k", "stress_qrpkl_seed3_10k"])
def test_fp64_matches_numpy_rts(name):
    """10,000 steps on three streams, FP64: x_smooth within 1e-9 of each state's max, var_smooth within 1e-9 of its max
    (SURVEY 8(c) norm).  Observed on a B200: default noise 5.9e-15 / 1.5e-13, stress (Q_R.pkl) noise 6.0e-14 / 2.8e-15."""
    _, kw, _ = cases.build(name)
    st = _streams(3, 10000, 11)
    res = kf_smooth(*_args(st), x0=kw["x0"], Q=kw["Q"], R=kw["R"], outputs=("x_smooth", "var_smooth"))
    ex, ev = _errors(res, st, kw, 3)
    print(f"{name}: x_smooth {ex:.2e}, var_smooth {ev:.2e}")
    assert ex <= 1e-9 and ev <= 1e-9
    assert int(res.status.max()) == 0


def test_fp32_within_stated_tolerance():
    """FP32, default noise, 10,000 steps on two streams: x_smooth within 2e-4 of each state's max, var_smooth within 2e-3 of its
    max.  Observed on a B200: 4.1e-6 / 6.6e-5, so the bounds leave a factor of ~30 for other inputs and builds."""
    _, kw, _ = cases.build("default_seed11_10k")
    st = _streams(2, 10000, 11)
    res = kf_smooth(*_args(st), x0=kw["x0"], Q=kw["Q"], R=kw["R"], dtype=torch.float32, outputs=("x_smooth", "var_smooth"))
    ex, ev = _errors(res, st, kw, 2)
    print(f"fp32: x_smooth {ex:.2e}, var_smooth {ev:.2e}")
    assert ex <= 2e-4 and ev <= 2e-3


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_last_step_is_the_filter(dtype):
    st = _streams(64, 120, 400)
    res = kf_smooth(*_args(st), dtype=dtype, outputs=("x_smooth", "var_smooth", "x_steps", "P_final"))
    assert torch.equal(res.x_smooth[-1], res.x_steps[-1])
    assert torch.equal(res.var_smooth[-1], res.P_final.reshape(12, 12, -1).diagonal(dim1=0, dim2=1).T)
    assert not torch.equal(res.x_smooth[0], res.x_steps[0])


def _forward_cases():
    S, T = 64, 200
    st = _streams(S, T, 500)
    N = 4 * S  # Monte-Carlo members sharing the streams, per-member Q / R
    q, r = monte_carlo_noise(np.arange(N), np.diag(cases.Q_DEFAULT), np.diag(cases.R_DEFAULT))
    idx = (np.arange(N) % S).astype(np.int32)
    return [
        ("streamed", st, dict(Q=q, R=r, n_traj=N)),
        ("direct", st, dict(Q=q, R=r, n_traj=N, stream_index=idx)),
        ("lone_warp", st, dict(n_traj=S)),
        ("packed_fp32", st, dict(Q=q, R=r, n_traj=N, dtype=torch.float32)),
        ("scalar_fp32", st, dict(Q=q, R=r, n_traj=N, dtype=torch.float32, packed=False)),
    ]


@pytest.mark.parametrize("case", range(5))
def test_forward_pass_is_kf_batch(case):
    """What the forward pass writes is bit-identical to kf_batch with the same arguments, on every SEQUENTIAL kernel."""
    name, st, kw = _forward_cases()[case]
    outs = ("x_steps", "summary")
    a = kf_batch(*_args(st), outputs=outs, truth=st["truth"], **kw)
    b = kf_smooth(*_args(st), outputs=outs + ("x_smooth",), truth=st["truth"], **kw)
    assert a.algo == b.algo == "sequential", name
    for o in outs:
        assert torch.equal(a.tensors[o], b.tensors[o]), (name, o)
    assert torch.equal(a.status, b.status), name
    assert torch.isfinite(b.x_smooth).all(), name
    # the smoother without x_steps among the outputs keeps x+ in its own storage and computes the same
    c = kf_smooth(*_args(st), outputs=("x_smooth",), **kw)
    assert torch.equal(b.x_smooth, c.x_smooth), name


def test_properties_variance_shrinks_and_degenerate_sizes():
    st = _streams(32, 100, 600)
    res = kf_smooth(*_args(st), outputs=("x_smooth", "var_smooth", "P_ckpt"), ckpt_every=1)
    diag_post = res.P_ckpt.reshape(100, 12, 12, -1).diagonal(dim1=1, dim2=2).permute(0, 2, 1)
    assert (res.var_smooth <= diag_post * (1 + 1e-9) + 1e-18).all()
    assert (res.var_smooth[:-1] < diag_post[:-1]).any()
    one = {k: v[:1] for k, v in st.items()}
    r1 = kf_smooth(*_args(one), outputs=("x_smooth", "var_smooth", "x_steps", "P_final"))
    assert torch.equal(r1.x_smooth, r1.x_steps)
    assert torch.equal(r1.var_smooth[0], r1.P_final.reshape(12, 12, -1).diagonal(dim1=0, dim2=1).T)
    zero = {k: v[:0] for k, v in st.items()}
    r0 = kf_smooth(*_args(zero), outputs=("x_smooth", "var_smooth", "summary"))
    assert r0.x_smooth.shape == (0, 12, 32) and r0.summary.shape[1] == 32
    rn = kf_smooth(*_args(st), n_traj=0, outputs=("x_smooth",))
    assert rn.x_smooth.shape == (100, 12, 0)


def test_singular_prior_sets_smooth_not_pd():
    """A group with zero P0 and zero Q (x, vx) keeps a zero prior covariance: its pivots are flagged, the filter's are not."""
    st = _streams(32, 50, 700)
    q = np.diag(cases.Q_DEFAULT).copy()
    q[[3, 9]] = 0.0
    res = kf_smooth(*_args(st), Q=q, P0=q, outputs=("x_smooth",))
    status = res.status.cpu().numpy()
    assert (status & 32).all() and not (status & 1).any()


def test_refusals_raise_value_error():
    st = _streams(4, 10, 800)
    dense_r = np.diag(cases.R_DEFAULT.diagonal()) + 1e-4 * (np.ones((10, 10)) - np.eye(10))
    coupled_p0 = cases.Q_DEFAULT.copy()
    coupled_p0[0, 3] = coupled_p0[3, 0] = 1e-4
    for kw, what in ((dict(cov_model="mpc", body_ref=st["truth"]), "predict"), (dict(structure="full"), "decoupled"),
                     (dict(R=dense_r), "diagonal"), (dict(P0=coupled_p0), "across the groups"), (dict(algo="joint"), "joint")):
        with pytest.raises(ValueError, match=what):
            kf_smooth(*_args(st), **kw)
