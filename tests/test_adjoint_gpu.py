"""GPU tests of the filter's adjoint (kf_vjp, kf_states): the CUDA adjoint kernel against the NumPy recursion of
tests/adjoint_oracle.py fed the GPU's own forward pass, on every forward kernel; shared inputs, FP32, the forward outputs,
gradcheck, the refusals, and a few Adam steps on simulated data with known truth."""
import numpy as np
import pytest
import torch

from oracle import cases
from oracle import kf_numpy as kn
from optistate_b200 import kf_batch, kf_measure, kf_states, kf_vjp
from optistate_b200.synth import make_streams, monte_carlo_noise
from tests import adjoint_oracle as ao

pytestmark = pytest.mark.gpu

FIELDS = (("q", slice(0, 12)), ("r", slice(12, 22)), ("x0", slice(22, 34)), ("P0", slice(34, 46)))


def _args(st):
    return st["imu"], st["p"], st["dp"], st["contact"], st["f"]


def _xbar(T, N, seed=3):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal((T, 12, N))).cuda()


def _per(v, n, N):
    v = np.asarray(v, float)
    return np.broadcast_to(v.reshape(n, -1), (n, N)) if v.ndim <= 1 or v.shape == (n,) else v


def _oracle(st, kw, xbar, members, stream_of, N):
    """Oracle grads [46, len(members)] fed the GPU forward pass (x+, x-, P+ from P_ckpt every step, z) of the same call."""
    z = kw.get("z")
    fw = kf_batch(*_args(st), outputs=("x_steps", "x_model_steps", "P_ckpt", "z_steps"), ckpt_every=1,
                  **{k: v for k, v in kw.items() if k != "z"}, z=z)
    xs, xm, Pc, zs = (fw.tensors[k].cpu().numpy() for k in ("x_steps", "x_model_steps", "P_ckpt", "z_steps"))
    T = xs.shape[0]
    q = _per(np.diag(cases.Q_DEFAULT) if kw.get("Q") is None else kw["Q"], 12, N)
    r = _per(np.diag(cases.R_DEFAULT) if kw.get("R") is None else kw["R"], 10, N)
    x0 = _per(cases.START if kw.get("x0") is None else kw["x0"], 12, N)
    P0 = kw.get("P0")
    xb = xbar.cpu().numpy()
    out = []
    for i in members:
        s = stream_of(i)
        C = ao.moments(st["p"][:, :, s], st["f"][:, :, s])
        p0 = np.diag(q[:, i]) if P0 is None else np.diag(_per(P0, 12, N)[:, i])
        out.append(ao.adjoint(xs[:, :, i], xm[:, :, i], Pc[:, :, i].reshape(T, 12, 12), zs[:, :, i], C, xb[:, :, i], x0[:, i], p0,
                              q[:, i], r[:, i]))
    return np.stack(out, axis=1)


def _errors(got, ref):
    return {name: float(np.abs(got[sl] - ref[sl]).max() / np.abs(ref[sl]).max()) for name, sl in FIELDS}


@pytest.mark.parametrize("noise,p0", [("default", None), ("default", "diag"), ("qrpkl", None), ("qrpkl", "diag")])
def test_fp64_matches_oracle_10k(noise, p0):
    """3 x 10,000 steps, FP64: every row group within 1e-9 of its largest magnitude (observed on a B200: at most 1.6e-15 with
    default noise, 3.8e-15 with Q_R.pkl noise)."""
    T, N = 10000, 3
    st = make_streams(range(11, 11 + N), T)
    Q, R = (cases.Q_DEFAULT, cases.R_DEFAULT) if noise == "default" else cases.q_r_pkl()
    kw = dict(Q=np.diag(Q).copy(), R=np.diag(R).copy(), x0=cases.START + np.r_[0.03, -0.02, 0.1, np.zeros(9)])
    if p0 == "diag":
        kw["P0"] = np.linspace(0.002, 0.03, 12)
    xbar = _xbar(T, N)
    res = kf_vjp(*_args(st), grad_x_steps=xbar, **kw)
    ref = _oracle(st, kw, xbar, range(N), lambda i: i, N)
    err = _errors(res.grad.cpu().numpy(), ref)
    print(noise, p0, err)
    assert max(err.values()) <= 1e-9, err
    assert int(res.status.max()) == 0


def _kernel_cases():
    S, T = 64, 200
    st = make_streams(range(500, 500 + S), T)
    N = 2 * S
    q, r = monte_carlo_noise(np.arange(N), np.diag(cases.Q_DEFAULT), np.diag(cases.R_DEFAULT))
    idx = ((np.arange(N) * 7) % S).astype(np.int32)
    z, _ = kf_measure(*(st[k] for k in ("imu", "p", "dp", "contact")))
    return st, [
        ("streamed", dict(Q=q, R=r, n_traj=N), lambda i: i % S, N),
        ("direct", dict(Q=q, R=r, n_traj=N, stream_index=idx), lambda i: int(idx[i]), N),
        ("lone_warp", dict(n_traj=S), lambda i: i, S),
        ("caller_z", dict(Q=q, R=r, n_traj=N, z=z), lambda i: i % S, N),
    ]


@pytest.mark.parametrize("case", range(4))
def test_each_forward_kernel(case):
    st, cases_ = _kernel_cases()
    name, kw, stream_of, N = cases_[case]
    xbar = _xbar(200, N, seed=case)
    res = kf_vjp(*_args(st), grad_x_steps=xbar, **kw)
    members = [0, 37, N - 1]
    ref = _oracle(st, kw, xbar, members, stream_of, N)
    err = _errors(res.grad.cpu().numpy()[:, members], ref)
    assert max(err.values()) <= 1e-9, (name, err)


def test_shared_and_per_trajectory_inputs():
    """Shared Q, R, x0 give the per-trajectory gradients of the same values; kf_states sums them over the trajectories."""
    S, T = 32, 100
    st = make_streams(range(900, 900 + S), T)
    q, r = np.diag(cases.Q_DEFAULT).copy(), np.diag(cases.R_DEFAULT).copy()
    x0 = cases.START + np.r_[0.05, 0.02, -0.1, np.zeros(9)]
    xbar = _xbar(T, S)
    a = kf_vjp(*_args(st), Q=q, R=r, x0=x0, grad_x_steps=xbar).grad
    b = kf_vjp(*_args(st), Q=np.repeat(q[:, None], S, 1), R=np.repeat(r[:, None], S, 1), x0=np.repeat(x0[:, None], S, 1),
               grad_x_steps=xbar).grad
    assert torch.equal(a, b)
    qt, rt, xt = (torch.tensor(v, device="cuda", requires_grad=True) for v in (q, r, x0))
    (kf_states(*_args(st), Q=qt, R=rt, x0=xt) * xbar).sum().backward()
    torch.testing.assert_close(qt.grad, a[0:12].sum(1) + a[34:46].sum(1), rtol=1e-12, atol=0)
    torch.testing.assert_close(rt.grad, a[12:22].sum(1), rtol=1e-12, atol=0)
    torch.testing.assert_close(xt.grad, a[22:34].sum(1), rtol=1e-12, atol=0)


def test_fp32_against_fp64():
    """T = 1,000, default noise: the FP32 gradient within 1e-4 of each row group's largest FP64 magnitude (observed on a B200:
    1.7e-6)."""
    S, T = 64, 1000
    st = make_streams(range(300, 300 + S), T)
    xbar = _xbar(T, S)
    g64 = kf_vjp(*_args(st), grad_x_steps=xbar).grad.cpu().numpy()
    g32 = kf_vjp(*_args(st), grad_x_steps=xbar.float(), dtype=torch.float32).grad.double().cpu().numpy()
    err = _errors(g32, g64)
    print("fp32", err)
    assert max(err.values()) <= 1e-4, err


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_forward_outputs_are_kf_batch(dtype):
    S, T = 64, 150
    st = make_streams(range(600, 600 + S), T)
    N = 3 * S
    q, r = monte_carlo_noise(np.arange(N), np.diag(cases.Q_DEFAULT), np.diag(cases.R_DEFAULT))
    kw = dict(Q=q, R=r, n_traj=N, dtype=dtype, truth=st["truth"])
    a = kf_batch(*_args(st), outputs=("x_steps", "summary"), **kw)
    b = kf_vjp(*_args(st), outputs=("x_steps", "summary"), grad_x_steps=_xbar(T, N).to(dtype), **kw)
    for o in ("x_steps", "summary"):
        assert torch.equal(a.tensors[o], b.tensors[o]), o
    assert torch.equal(a.status, b.status)
    c = kf_states(*_args(st), Q=torch.tensor(q, device="cuda", dtype=dtype), R=r, n_traj=N, dtype=dtype)
    assert torch.equal(c, a.x_steps)


def test_gradcheck_kf_states():
    S, T = 3, 50
    st = {k: torch.from_numpy(v).cuda() for k, v in make_streams(range(700, 700 + S), T).items()}
    q = torch.tensor(np.repeat(np.diag(cases.Q_DEFAULT)[:, None], S, 1), device="cuda", requires_grad=True)
    r = torch.tensor(np.diag(cases.R_DEFAULT), device="cuda", requires_grad=True)
    x0 = torch.tensor(np.repeat((cases.START + np.r_[0.1, -0.05, 0.2, np.zeros(9)])[:, None], S, 1), device="cuda", requires_grad=True)
    p0 = torch.tensor(np.linspace(0.002, 0.03, 12), device="cuda", requires_grad=True)
    fn = lambda q, r, x0, p0: kf_states(*_args(st), x0=x0, P0=p0, Q=q, R=r)  # noqa: E731
    assert torch.autograd.gradcheck(fn, (q, r, x0, p0), eps=1e-6, atol=1e-6, rtol=1e-4, fast_mode=True)


def test_refusals_raise_value_error():
    st = make_streams(range(800, 804), 10)
    xbar = _xbar(10, 4)
    dense_r = cases.R_DEFAULT + 1e-4 * (np.ones((10, 10)) - np.eye(10))
    coupled_p0 = cases.Q_DEFAULT.copy()
    coupled_p0[0, 3] = coupled_p0[3, 0] = 1e-4
    for kw, what in ((dict(cov_model="mpc", body_ref=st["truth"]), "predict"), (dict(structure="full"), "decoupled"),
                     (dict(R=dense_r), "diagonal"), (dict(P0=coupled_p0), "across the groups"), (dict(algo="joint"), "joint")):
        with pytest.raises(ValueError, match=what):
            kf_vjp(*_args(st), grad_x_steps=xbar, **kw)
        with pytest.raises(ValueError, match=what):
            kf_states(*_args(st), **kw)
    block_p0 = cases.Q_DEFAULT.copy()
    block_p0[0, 6] = block_p0[6, 0] = 1e-4  # dense, inside {th, w}: taken by kf_vjp, refused by kf_states when it requires grad
    assert kf_vjp(*_args(st), P0=block_p0, grad_x_steps=xbar).grad.shape == (46, 4)
    with pytest.raises(ValueError, match="dense P0"):
        kf_states(*_args(st), P0=torch.tensor(block_p0, device="cuda", requires_grad=True))


def _simulate(st, q_true, r_true, x0, seed=5, dt=kn.DT):
    """Truth from the kernels' mean model with process noise q_true, and z = H x + noise r_true: x [T, 12, S], z [T, 10, S]."""
    T, S = st["p"].shape[0], st["p"].shape[2]
    rng = np.random.default_rng(seed)
    xs, zs = np.empty((T, 12, S)), np.empty((T, 10, S))
    d = dt / kn.INERTIA
    for s in range(S):
        x = x0.copy()
        C = ao.moments(st["p"][:, :, s], st["f"][:, :, s]).reshape(-1, 3, 3)
        fs = st["f"][:, :, s].reshape(-1, 4, 3).sum(axis=1)
        for t in range(T):
            R = kn.rot_zyx(*x[0:3])
            CR = C[t] @ R
            g = np.array([CR[1, 2] - CR[2, 1], CR[2, 0] - CR[0, 2], CR[0, 1] - CR[1, 0]])
            xn = x.copy()
            xn[0:3] = x[0:3] + dt * (np.trunc(R.T) @ x[6:9])
            xn[3:6] = x[3:6] + dt * x[9:12]
            xn[6:9] = x[6:9] + R @ (d * g)
            xn[9:12] = x[9:12] + (dt / kn.MASS) * fs[t]
            xn[11] += dt * kn.GRAVITY
            x = xn + np.sqrt(q_true) * rng.standard_normal(12)
            xs[t, :, s] = x
            zs[t, :, s] = x[kn.SEL] + np.sqrt(r_true) * rng.standard_normal(10)
    return xs, zs


def test_adam_on_log_noise_lowers_rmse_against_truth():
    """Data simulated from the mean model with known truth: 30 Adam steps on log q and log r through kf_states, from a start
    100 times off, lower the RMSE of x_steps against the truth.  q of x and y reaches only P_xx (P_yy), which no gain reads, so
    x_steps does not depend on it: its gradient is exactly zero, while every other entry of q gets one."""
    S, T = 32, 300
    st = make_streams(range(1000, 1000 + S), T)
    q_true = np.diag(cases.Q_DEFAULT) * 1e-2
    r_true = np.diag(cases.R_DEFAULT)
    x0 = cases.START + np.r_[0.05, -0.02, 0.1, np.zeros(9)]
    truth, z = _simulate(st, q_true, r_true, x0)
    truth, z = torch.from_numpy(truth).cuda(), torch.from_numpy(z).cuda()
    lq = torch.tensor(np.log(q_true * 100), device="cuda", requires_grad=True)
    lr = torch.tensor(np.log(r_true / 100), device="cuda", requires_grad=True)
    opt = torch.optim.Adam([lq, lr], lr=0.2)
    rmse = []
    for k in range(31):
        xs = kf_states(None, st["p"], None, None, st["f"], x0=x0, Q=lq.exp(), R=lr.exp(), z=z)
        loss = ((xs - truth) ** 2).mean()
        rmse.append(float(loss.detach().sqrt()))
        opt.zero_grad()
        loss.backward()
        if k == 0:
            assert (lq.grad[[3, 4]] == 0).all() and (lq.grad[[0, 1, 2, 5, 6, 7, 8, 9, 10, 11]] != 0).all(), lq.grad
        opt.step()
    print("rmse", rmse[0], rmse[-1])
    assert rmse[-1] < rmse[0], rmse


@pytest.mark.parametrize("N", [12, 10])
def test_diagonal_matrix_inputs_with_n_trajectories_equal_to_n(N):
    """A shared diagonal-matrix Q, R or P0 ([n, n]) is passed on as a shared diagonal, so its gradient is the diagonal matrix of
    the per-trajectory gradients summed, also when N equals n (12 for Q and P0, 10 for R) and the shape alone would read as
    [n, N]."""
    st = make_streams(range(1100, 1100 + N), 60)
    q, r, p0 = np.diag(cases.Q_DEFAULT).copy(), np.diag(cases.R_DEFAULT).copy(), np.linspace(0.002, 0.03, 12)
    xbar = _xbar(60, N)
    g = kf_vjp(*_args(st), Q=q, R=r, P0=p0, grad_x_steps=xbar).grad
    qt, rt, pt = (torch.tensor(np.diag(v), device="cuda", requires_grad=True) for v in (q, r, p0))
    (kf_states(*_args(st), Q=qt, R=rt, P0=pt) * xbar).sum().backward()
    for t, sl in ((qt, slice(0, 12)), (rt, slice(12, 22)), (pt, slice(34, 46))):
        assert t.grad.shape == t.shape
        torch.testing.assert_close(t.grad, torch.diag(g[sl].sum(1)), rtol=1e-12, atol=0)
    # the same values per trajectory: [n, N] gradients as they are
    qn = torch.tensor(np.repeat(q[:, None], N, 1), device="cuda", requires_grad=True)
    (kf_states(*_args(st), Q=qn, R=r, P0=p0, q_kind=2) * xbar).sum().backward()
    torch.testing.assert_close(qn.grad, g[0:12], rtol=1e-12, atol=0)


def test_input_changed_in_place_before_backward_raises():
    st = make_streams(range(1200, 1204), 20)
    q = torch.tensor(np.diag(cases.Q_DEFAULT), device="cuda", requires_grad=True)
    qe = q * 1.0
    xs = kf_states(*_args(st), Q=qe)
    with torch.no_grad():
        qe.mul_(2.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        xs.sum().backward()


def test_bad_pivot_warns():
    """Zero process noise, initial variance and measurement noise of vx: the pivot of that measurement is 0 in the filter and in
    the adjoint, and kf_states warns on the backward pass."""
    st = make_streams(range(1300, 1304), 20)
    q = np.diag(cases.Q_DEFAULT).copy()
    q[[3, 9]] = 0.0
    r = np.diag(cases.R_DEFAULT).copy()
    r[7] = 0.0
    rt = torch.tensor(r, device="cuda", requires_grad=True)
    xs = kf_states(*_args(st), Q=q, P0=q, R=rt)
    with pytest.warns(RuntimeWarning, match="non-zero status"):
        xs.sum().backward()
