"""GPU tests of the full-covariance smoother (kf_smooth_full): the dense backward kernel against the NumPy recursion of
tests/rts_full_oracle.py on the GPU's own forward pass, end to end against the NumPy filter, against kf_smooth where both apply,
its forward pass against kf_batch, the closed loop's output, FP32, and its properties and refusals."""
import numpy as np
import pytest
import torch

from oracle import cases
from optistate_b200 import kf_batch, kf_smooth, kf_smooth_full
from optistate_b200.synth import make_streams
from tests import rts_full_oracle as rf

pytestmark = pytest.mark.gpu


def _args(st):
    return st["imu"], st["p"], st["dp"], st["contact"], st["f"]


def _coupled_p0():
    rng = np.random.default_rng(77)
    A = rng.standard_normal((12, 12))
    return 0.02 * (A @ A.T / 12 + 0.5 * np.eye(12))


def _setup(name):
    """(kwargs of kf_smooth_full, model): predict with a coupled SPD P0, or the predict_mpc model (body_ref = truth)."""
    if name == "predict_coupled_p0":
        return dict(P0=_coupled_p0(), Q=cases.Q_DEFAULT, R=cases.R_DEFAULT), "predict"
    if name == "mpc_default":
        return dict(Q=cases.Q_DEFAULT, R=cases.R_DEFAULT, cov_model="mpc"), "mpc"
    q, r = cases.q_r_pkl()
    return dict(Q=q, R=r, cov_model="mpc"), "mpc"


def _backward_errors(res, st, kw, model, n, T):
    """Largest error of x_smooth and var_smooth, relative to each state's largest value, of the CUDA backward kernel against the
    NumPy recursion run on the GPU's own forward pass (x_steps, x_model_steps, P_ckpt every step)."""
    x_post = res.x_steps.cpu().numpy()
    x_prior = res.x_model_steps.cpu().numpy()
    P_post = res.P_ckpt.cpu().numpy().reshape(T, 12, 12, -1)
    xs_g, vs_g = res.x_smooth.cpu().numpy().astype(np.float64), res.var_smooth.cpu().numpy().astype(np.float64)
    Q = np.diag(np.diag(np.asarray(kw["Q"], float)))
    ex = ev = 0.0
    for j in range(n):
        F = rf.transitions(x_post[:, :, j], model, st["body_ref"][:, :, j] if model == "mpc" else None, cases.START)
        xs, Ps = rf.rts(x_post[:, :, j], x_prior[:, :, j], np.ascontiguousarray(P_post[:, :, :, j]), Q, F)
        e = rf.rel_errors(xs_g[:, :, j], vs_g[:, :, j], xs, np.einsum("tii->ti", Ps))
        ex, ev = max(ex, e[0]), max(ev, e[1])
    return ex, ev


@pytest.mark.parametrize("name,bound", [("predict_coupled_p0", 1e-9), ("mpc_default", 1e-9), ("mpc_qrpkl", 5e-8)])
def test_backward_matches_numpy_on_the_gpu_forward_pass(name, bound):
    """3 streams x 10,000 steps, FP64.  mpc + Q_R.pkl: cond(P-) ~5e7, and two FP64 NumPy solvers of the same recursion already
    differ by 6.8e-9 there (tests/test_smooth_full_cpu.py), so its bound is looser.  Observed on a B200: predict + coupled P0
    5.3e-15 / 1.5e-13, mpc 3.8e-15 / 1.8e-15, mpc + Q_R.pkl 6.0e-10 / 1.8e-10 (x_smooth / var_smooth)."""
    kw, model = _setup(name)
    T = 10000
    st = make_streams(range(11, 14), T)
    if model == "mpc":
        kw = dict(kw, body_ref=st["truth"])
    res = kf_smooth_full(*_args(st), outputs=("x_smooth", "var_smooth", "x_steps", "x_model_steps", "P_ckpt"), ckpt_every=1, **kw)
    if model == "mpc":
        st = dict(st, body_ref=st["truth"])
    ex, ev = _backward_errors(res, st, kw, model, 3, T)
    print(f"{name}: x_smooth {ex:.2e}, var_smooth {ev:.2e}")
    assert ex <= bound and ev <= bound
    assert int(res.status.max()) == 0


def test_end_to_end_next_mpc_cov_seed5():
    """The predict_mpc case whose filter is pinned to the unmodified reference (tests/test_parity_gpu.py), 400 steps: kf_smooth_full
    against the NumPy filter + recursion of the same model.  Its noise is Q_R.pkl, where cond(P-) ~5e7 amplifies the two forward
    passes' own difference (sequential against joint update, ~1e-11 of P) and where the NumPy recursion's variances are only good
    to ~4e-5 against the dense certificate (DESIGN.md section 0.2).  Observed on a B200: x_smooth 4.4e-8, var_smooth 4.2e-5; the
    bounds leave a factor of ~10."""
    stream, kw, _ = cases.build("next_mpc_cov_seed5")
    s = cases.stack_stream(stream)
    res = kf_smooth_full(s["imu"], s["p"], s["dp"], s["contact"], s["f"], x0=kw["x0"], Q=kw["Q"], R=kw["R"], cov_model="mpc",
                         body_ref=s["body_ref"], outputs=("x_smooth", "var_smooth"))
    fw = rf.forward(stream, kw["x0"], kw["P0"], kw["Q"], kw["R"], "mpc")
    xs, Ps = rf.rts(fw["x"], fw["x_model"], fw["P"], kw["Q"], fw["F"])
    ex, ev = rf.rel_errors(res.x_smooth[:, :, 0].cpu().numpy(), res.var_smooth[:, :, 0].cpu().numpy(), xs, np.einsum("tii->ti", Ps))
    print(f"next_mpc_cov_seed5: x_smooth {ex:.2e}, var_smooth {ev:.2e}")
    assert ex <= 5e-7 and ev <= 5e-4


@pytest.mark.parametrize("case", ["default", "diag_p0", "block_p0"])
def test_equals_kf_smooth_where_both_apply(case):
    st = make_streams(range(900, 964), 300)
    kw = {}
    if case == "diag_p0":
        _, ckw, _ = cases.build("edge_diag_p0_seed31")
        kw = dict(P0=ckw["P0"], Q=ckw["Q"], R=ckw["R"])
    elif case == "block_p0":
        _, ckw, _ = cases.build("edge_block_p0_seed32")
        kw = dict(P0=ckw["P0"])
    a = kf_smooth(*_args(st), outputs=("x_smooth", "var_smooth"), **kw)
    b = kf_smooth_full(*_args(st), outputs=("x_smooth", "var_smooth"), **kw)
    for o in ("x_smooth", "var_smooth"):
        x, y = a.tensors[o], b.tensors[o]
        scale = x.abs().amax(dim=(0, 2), keepdim=True).clamp_min(1e-300)
        err = float(((x - y).abs() / scale).max())
        print(f"{case} {o}: {err:.2e}")
        assert err <= 1e-12, (case, o, err)


def _forward_cases():
    S, T = 64, 150
    st = make_streams(range(500, 500 + S), T)
    N = 2 * S
    q = np.tile(np.diag(cases.Q_DEFAULT)[:, None], (1, N)) * np.linspace(0.5, 2.0, N)[None, :]
    idx = (np.arange(N) % S).astype(np.int32)
    mpc = dict(cov_model="mpc", body_ref=st["truth"])
    return st, [
        ("streamed", dict(Q=q, n_traj=N)),
        ("streamed_coupled_p0", dict(P0=_coupled_p0(), n_traj=N)),
        ("direct", dict(Q=q, n_traj=N, stream_index=idx)),
        ("lone_warp", dict(n_traj=S)),
        ("packed_fp32", dict(Q=q, n_traj=N, dtype=torch.float32)),
        ("scalar_fp32", dict(Q=q, n_traj=N, dtype=torch.float32, packed=False)),
        ("mpc_streamed", dict(Q=q, n_traj=N, **mpc)),
        ("mpc_direct", dict(Q=q, n_traj=N, stream_index=idx, **mpc)),
        ("mpc_packed_fp32", dict(n_traj=N, dtype=torch.float32, **mpc)),
        ("mpc_scalar_fp32", dict(n_traj=N, dtype=torch.float32, packed=False, **mpc)),
    ]


@pytest.mark.parametrize("case", range(10))
def test_forward_pass_is_kf_batch(case):
    """x_steps, summary and status of the forward pass are bit-identical to kf_batch with the same arguments (which runs the
    decoupled-group kernels where they apply: the full ones match them bit for bit)."""
    st, cs = _forward_cases()
    name, kw = cs[case]
    outs = ("x_steps", "summary")
    a = kf_batch(*_args(st), outputs=outs, truth=st["truth"], **kw)
    b = kf_smooth_full(*_args(st), outputs=outs + ("x_smooth",), truth=st["truth"], **kw)
    assert a.algo == b.algo == "sequential", name
    for o in outs:
        assert torch.equal(a.tensors[o], b.tensors[o]), (name, o)
    assert torch.equal(a.status, b.status), name
    assert torch.isfinite(b.x_smooth).all(), name


def test_closed_loop_output_smoothed():
    """estimate_state_mpc_batch (64 trajectories x 100 steps, the reference set-up of tests/test_mpc_gpu.py): kf_batch with its
    forces and the predict_mpc model reproduces its x_steps bit for bit (each closed-loop step is one optistate_kf_batch call of the
    same kernel, with P handed over exactly); kf_smooth_full on the same ends at the filter and shrinks every variance."""
    from optistate_b200.mpc import estimate_state_mpc_batch

    T, N = 100, 64
    st = make_streams(range(N), T)
    rng = np.random.default_rng(4)
    ref = np.zeros((T, 5, 12, N))
    ref[:, :, 5, :] = 0.28
    ref[:, :, 0:3, :] = 0.02 * rng.standard_normal((T, 5, 3, N))
    xs, fs, mst, fst = estimate_state_mpc_batch(st["imu"], st["p"], st["dp"], st["contact"], ref)
    body_ref = np.ascontiguousarray(ref[:, 0])
    a = kf_batch(st["imu"], st["p"], st["dp"], st["contact"], fs, cov_model="mpc", body_ref=body_ref, n_traj=N, outputs=("x_steps",))
    assert torch.equal(a.x_steps, xs)
    res = kf_smooth_full(st["imu"], st["p"], st["dp"], st["contact"], fs, cov_model="mpc", body_ref=body_ref, n_traj=N,
                         outputs=("x_smooth", "var_smooth", "P_ckpt"), ckpt_every=1)
    assert torch.equal(res.x_smooth[-1], xs[-1])
    diag_post = res.P_ckpt.reshape(T, 12, 12, -1).diagonal(dim1=1, dim2=2).permute(0, 2, 1)
    assert (res.var_smooth <= diag_post * (1 + 1e-9) + 1e-18).all()
    assert (res.var_smooth[:-1] < diag_post[:-1]).any()
    assert int(res.status.max()) == 0


@pytest.mark.parametrize("name", ["predict_coupled_p0", "mpc_default"])
def test_fp32_within_stated_tolerance(name):
    """FP32, default noise, 2 streams x 10,000 steps, against the FP64 NumPy recursion on the FP32 forward pass.  Bounds: x_smooth
    2e-4 and var_smooth 2e-3 of each state's largest value.  Observed on a B200: predict + coupled P0 4.3e-6 / 3.7e-5, mpc 4.5e-7 /
    7.7e-7, so the bounds leave a factor of ~50 or more."""
    kw, model = _setup(name)
    T = 10000
    st = make_streams(range(11, 13), T)
    if model == "mpc":
        kw = dict(kw, body_ref=st["truth"])
    res = kf_smooth_full(*_args(st), dtype=torch.float32, outputs=("x_smooth", "var_smooth", "x_steps", "x_model_steps", "P_ckpt"),
                         ckpt_every=1, **kw)
    if model == "mpc":
        st = dict(st, body_ref=st["truth"])
    ex, ev = _backward_errors(res, st, kw, model, 2, T)
    print(f"fp32 {name}: x_smooth {ex:.2e}, var_smooth {ev:.2e}")
    assert ex <= 2e-4 and ev <= 2e-3


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_properties_and_degenerate_sizes(dtype):
    st = make_streams(range(600, 632), 100)
    kw = dict(cov_model="mpc", body_ref=st["truth"])
    res = kf_smooth_full(*_args(st), dtype=dtype, outputs=("x_smooth", "var_smooth", "x_steps", "P_final", "P_ckpt"), ckpt_every=1, **kw)
    assert torch.equal(res.x_smooth[-1], res.x_steps[-1])
    assert torch.equal(res.var_smooth[-1], res.P_final.reshape(12, 12, -1).diagonal(dim1=0, dim2=1).T)
    assert not torch.equal(res.x_smooth[0], res.x_steps[0])
    diag_post = res.P_ckpt.reshape(100, 12, 12, -1).diagonal(dim1=1, dim2=2).permute(0, 2, 1)
    slack = 1e-9 if dtype == torch.float64 else 1e-4
    assert (res.var_smooth <= diag_post * (1 + slack) + 1e-18).all()
    one = {k: v[:1] for k, v in st.items()}
    r1 = kf_smooth_full(*_args(one), dtype=dtype, outputs=("x_smooth", "var_smooth", "x_steps", "P_final"), cov_model="mpc",
                        body_ref=one["truth"])
    assert torch.equal(r1.x_smooth, r1.x_steps)
    assert torch.equal(r1.var_smooth[0], r1.P_final.reshape(12, 12, -1).diagonal(dim1=0, dim2=1).T)
    zero = {k: v[:0] for k, v in st.items()}
    r0 = kf_smooth_full(*_args(zero), dtype=dtype, outputs=("x_smooth", "var_smooth", "summary"), cov_model="mpc", body_ref=zero["truth"])
    assert r0.x_smooth.shape == (0, 12, 32) and r0.summary.shape[1] == 32
    rn = kf_smooth_full(*_args(st), dtype=dtype, n_traj=0, outputs=("x_smooth",), **kw)
    assert rn.x_smooth.shape == (100, 12, 0)
    # N not a multiple of the 32 trajectories of a block: the spare lanes store nothing
    r5 = kf_smooth_full(*_args(st), dtype=dtype, n_traj=37, outputs=("x_smooth",), **kw)
    r5b = kf_smooth_full(*_args(st), dtype=dtype, n_traj=64, outputs=("x_smooth",), **kw)
    assert torch.equal(r5.x_smooth, r5b.x_smooth[:, :, :37])


def test_singular_prior_sets_smooth_not_pd():
    """A zero row of Q and P0 (x and vx) keeps a zero prior variance under the predict() model: the smoother's pivot is flagged,
    the filter's is not (x is not measured)."""
    st = make_streams(range(700, 732), 50)
    q = np.diag(cases.Q_DEFAULT).copy()
    q[[3, 9]] = 0.0
    P0 = _coupled_p0()
    P0[[3, 9], :] = 0.0
    P0[:, [3, 9]] = 0.0
    res = kf_smooth_full(*_args(st), Q=q, P0=P0, outputs=("x_smooth",))
    status = res.status.cpu().numpy()
    assert (status & 32).all() and not (status & 1).any()


def test_refusals_raise_value_error():
    st = make_streams(range(800, 804), 10)
    dense_r = np.diag(cases.R_DEFAULT.diagonal()) + 1e-4 * (np.ones((10, 10)) - np.eye(10))
    nonsym = _coupled_p0()
    nonsym[0, 3] += 1e-4
    for kw, what in ((dict(algo="joint"), "joint"), (dict(R=dense_r), "diagonal"), (dict(P0=nonsym), "symmetric")):
        with pytest.raises(ValueError, match=what):
            kf_smooth_full(*_args(st), **kw)
