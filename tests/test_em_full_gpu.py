"""GPU tests of the E-step on the full covariance (kf_noise_stats_full) and its EM loop (kf_noise_em_full): the CUDA statistics
against tests/em_oracle.py's textbook E-step fed the GPU's own forward pass, FP32, the smoothed and forward outputs against
kf_smooth_full / kf_batch, kf_noise_stats where both apply, degenerate sizes, status and refusals, the EM loop against NumPy, and
the closed loop's output."""
import numpy as np
import pytest
import torch

from oracle import cases
from oracle import kf_numpy as kn
from optistate_b200 import kf_batch, kf_noise_em_full, kf_noise_stats, kf_noise_stats_full, kf_smooth_full
from optistate_b200 import _native as nv
from optistate_b200.batch import kf_measure
from optistate_b200.synth import make_streams, monte_carlo_noise
from tests import em_full_oracle as ef
from tests import em_oracle as eo
from tests import rts_full_oracle as rf
from tests.test_smooth_full_gpu import _coupled_p0, _forward_cases, _setup

pytestmark = pytest.mark.gpu


def _args(st):
    return st["imu"], st["p"], st["dp"], st["contact"], st["f"]


def _rel(a, b):
    return float((np.abs(a - b) / np.abs(b)).max())


def _gpu_chain_stats(st, kw, model, n, T, dtype=torch.float64):
    """(GPU noise_stats [23, n], NumPy textbook E-step [23, n] on the GPU's own forward pass: x_steps, x_model_steps, P_ckpt every
    step and the GPU's z)."""
    kw = dict(kw, body_ref=st["truth"]) if model == "mpc" else kw
    res = kf_noise_stats_full(*_args(st), dtype=dtype, outputs=("x_steps", "x_model_steps", "P_ckpt"), ckpt_every=1, **kw)
    z, _ = kf_measure(st["imu"], st["p"], st["dp"], st["contact"], dtype=dtype)
    z = z.cpu().numpy().astype(np.float64)
    x_post, x_prior = res.x_steps.cpu().numpy().astype(np.float64), res.x_model_steps.cpu().numpy().astype(np.float64)
    P_post = res.P_ckpt.cpu().numpy().astype(np.float64).reshape(T, 12, 12, -1)
    Q, R = np.diag(np.diag(np.asarray(kw["Q"], float))), np.diag(np.diag(np.asarray(kw["R"], float)))
    P0 = Q if kw.get("P0") is None else np.asarray(kw["P0"], float)
    ref = np.empty((23, n))
    for j in range(n):
        F = rf.transitions(x_post[:, :, j], model, st["truth"][:, :, j] if model == "mpc" else None, cases.START)
        ch = dict(Xp=np.concatenate([cases.START.reshape(1, 12), x_post[:, :, j]]), PP=np.concatenate([P0[None], P_post[..., j]]),
                  xm=x_prior[:, :, j], Fs=F, z=z[:, :, j])
        Sw, Sv, ll = eo.estep_textbook(ch, Q, R)
        ref[:12, j], ref[12:22, j], ref[22, j] = Sw, Sv, ll
    return res, res.noise_stats.cpu().numpy().astype(np.float64), ref


@pytest.mark.parametrize("name,bound", [("predict_coupled_p0", 1e-9), ("mpc_default", 1e-9), ("mpc_qrpkl", 5e-8)])
def test_fp64_matches_numpy_on_the_gpu_forward_pass(name, bound):
    """3 streams x 10,000 steps, FP64, every Sw / Sv row and the log-likelihood relative to NumPy.  mpc + Q_R.pkl: cond(P-) ~5e7,
    where two FP64 solvers of the NumPy recursion already differ by 1.5e-9 in Sw over 2,000 steps (tests/test_em_full_cpu.py), so
    its bound is looser.  Observed errors are printed and quoted in DESIGN.md section 0.3."""
    kw, model = _setup(name)
    T = 10000
    st = make_streams(range(11, 14), T)
    res, got, ref = _gpu_chain_stats(st, kw, model, 3, T)
    e = [_rel(got[a:b], ref[a:b]) for a, b in ((0, 12), (12, 22), (22, 23))]
    print(f"{name}: Sw {e[0]:.2e}, Sv {e[1]:.2e}, loglik {e[2]:.2e}")
    assert max(e) <= bound
    assert int(res.status.max()) == 0


@pytest.mark.parametrize("name", ["predict_coupled_p0", "mpc_default"])
def test_fp32_within_stated_tolerance(name):
    """FP32, default noise, 2 streams x 10,000 steps, against NumPy on the FP32 forward pass.  Bounds as for kf_noise_stats: Sw / Sv
    2e-2 relative, log-likelihood 1e-3."""
    kw, model = _setup(name)
    T = 10000
    st = make_streams(range(11, 13), T)
    _, got, ref = _gpu_chain_stats(st, kw, model, 2, T, torch.float32)
    es, el = _rel(got[:22], ref[:22]), _rel(got[22], ref[22])
    print(f"fp32 {name}: stats {es:.2e}, loglik {el:.2e}")
    assert es <= 2e-2 and el <= 1e-3


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_smoothed_outputs_are_kf_smooth_full(dtype):
    st = make_streams(range(900, 964), 150)
    for kw in (dict(P0=_coupled_p0()), dict(cov_model="mpc", body_ref=st["truth"])):
        a = kf_smooth_full(*_args(st), dtype=dtype, outputs=("x_smooth", "var_smooth"), **kw)
        b = kf_noise_stats_full(*_args(st), dtype=dtype, outputs=("x_smooth", "var_smooth"), **kw)
        assert torch.equal(a.x_smooth, b.x_smooth) and torch.equal(a.var_smooth, b.var_smooth)
        assert torch.isfinite(b.noise_stats).all()


@pytest.mark.parametrize("case", range(10))
def test_forward_pass_is_kf_batch(case):
    st, cs = _forward_cases()
    name, kw = cs[case]
    outs = ("x_steps", "summary")
    a = kf_batch(*_args(st), outputs=outs, truth=st["truth"], **kw)
    b = kf_noise_stats_full(*_args(st), outputs=outs, truth=st["truth"], **kw)
    assert b.algo == "sequential", name
    for o in outs:
        assert torch.equal(a.tensors[o], b.tensors[o]), (name, o)
    assert torch.equal(a.status, b.status), name
    assert torch.isfinite(b.noise_stats).all(), name


@pytest.mark.parametrize("case", ["default", "block_p0"])
def test_equals_kf_noise_stats_where_both_apply(case):
    st = make_streams(range(900, 964), 300)
    kw = {}
    if case == "block_p0":
        _, ckw, _ = cases.build("edge_block_p0_seed32")
        kw = dict(P0=ckw["P0"])
    a = kf_noise_stats(*_args(st), **kw).noise_stats
    b = kf_noise_stats_full(*_args(st), **kw).noise_stats
    err = float(((a - b).abs() / a.abs()).max())
    print(f"{case}: {err:.2e}")
    assert err <= 1e-12


def test_degenerate_sizes():
    st = make_streams(range(600, 632), 100)
    kw = dict(cov_model="mpc", body_ref=st["truth"])
    # N not a multiple of the 32 trajectories of a block: the spare lanes store nothing
    r5 = kf_noise_stats_full(*_args(st), n_traj=37, outputs=("x_smooth",), **kw)
    r5b = kf_noise_stats_full(*_args(st), n_traj=64, outputs=("x_smooth",), **kw)
    assert torch.equal(r5.noise_stats, r5b.noise_stats[:, :37]) and torch.equal(r5.x_smooth, r5b.x_smooth[:, :, :37])
    one = {k: v[:1] for k, v in st.items()}  # T = 1: the t = -1 transition and the first measurement only
    for name in ("predict_coupled_p0", "mpc_default"):
        kw1, model = _setup(name)
        _, got, ref = _gpu_chain_stats(one, kw1, model, 32, 1)
        assert _rel(got, ref) <= 1e-9, name
    zero = {k: v[:0] for k, v in st.items()}
    r0 = kf_noise_stats_full(*_args(zero), cov_model="mpc", body_ref=zero["truth"])
    assert r0.noise_stats.shape == (23, 32) and not r0.noise_stats.any()
    rn = kf_noise_stats_full(*_args(st), n_traj=0, outputs=("x_smooth",), **kw)
    assert rn.noise_stats.shape == (23, 0) and rn.x_smooth.shape == (100, 12, 0)


def test_singular_prior_sets_smooth_not_pd_and_bad_innovation_gives_nan():
    st = make_streams(range(700, 732), 50)
    q = np.diag(cases.Q_DEFAULT).copy()
    q[[3, 9]] = 0.0
    P0 = _coupled_p0()
    P0[[3, 9], :] = 0.0
    P0[:, [3, 9]] = 0.0
    res = kf_noise_stats_full(*_args(st), Q=q, P0=P0)
    status = res.status.cpu().numpy()
    assert (status & 32).all() and not (status & 1).any()
    # vx (measurement row 7) keeps a zero prior variance: with r = 0 the innovation pivot is 0 and the log-likelihood NaN
    r = np.diag(cases.R_DEFAULT).copy()
    r[7] = 0.0
    res = kf_noise_stats_full(*_args(st), Q=q, P0=P0, R=r)
    assert torch.isnan(res.noise_stats[22]).all()


def test_refusals_raise_value_error():
    st = make_streams(range(800, 804), 10)
    dense_r = np.diag(cases.R_DEFAULT.diagonal()) + 1e-4 * (np.ones((10, 10)) - np.eye(10))
    nonsym = _coupled_p0()
    nonsym[0, 3] += 1e-4
    dense_q = cases.Q_DEFAULT + 1e-6 * (np.ones((12, 12)) - np.eye(12))
    for kw, what in ((dict(algo="joint"), "joint"), (dict(R=dense_r), "diagonal"), (dict(Q=dense_q), "diagonal"),
                     (dict(P0=nonsym), "symmetric")):
        with pytest.raises(ValueError, match=what):
            kf_noise_stats_full(*_args(st), **kw)
    with pytest.raises(ValueError, match="diagonal"):
        kf_noise_em_full(*_args(st), R=dense_r, iters=1)


def _simulated(S, T, seed0=0):
    sims = [eo.simulate(seed0 + j, T, kn.Q_DEFAULT * 0.5, kn.R_DEFAULT * 2.0) for j in range(S)]
    st = {k: np.ascontiguousarray(np.stack([s[0][k] for s in sims], axis=-1)) for k in sims[0][0]}
    z = np.ascontiguousarray(np.stack([s[1] for s in sims], axis=-1))
    return sims, st, z


def test_em_matches_numpy_shared_and_per_member():
    """5 iterations under predict_mpc on 4 simulated streams: Q, R and the log-likelihood equal the NumPy EM loop to 1e-8 relative,
    pooled, and per trajectory for Monte-Carlo members that share the streams and start from different Q / R."""
    sims, st, z = _simulated(4, 200)
    streams = [dict(s[0], body_ref=s[0]["truth"]) for s in sims]
    res = kf_noise_em_full(*_args(st), z=z, iters=5, shared=True, cov_model="mpc", body_ref=st["truth"])
    q, r, ll = ef.em(streams, kn.Q_DEFAULT, kn.R_DEFAULT, 5, True, zs=[s[1] for s in sims], model="mpc")
    assert _rel(res.Q.cpu().numpy(), q) <= 1e-8 and _rel(res.R.cpu().numpy(), r) <= 1e-8
    assert _rel(res.loglik.cpu().numpy(), ll) <= 1e-8
    N = 8
    q0, r0 = monte_carlo_noise(np.arange(N), kn.Q_DEFAULT, kn.R_DEFAULT)
    idx = (np.arange(N) % 4).astype(np.int32)
    res = kf_noise_em_full(*_args(st), Q=q0, R=r0, z=z, iters=5, n_traj=N, stream_index=idx, cov_model="mpc", body_ref=st["truth"])
    q, r, ll = ef.em([streams[j] for j in idx], q0.T, r0.T, 5, False, zs=[sims[j][1] for j in idx], model="mpc")
    assert _rel(res.Q.cpu().numpy(), q.T) <= 1e-8 and _rel(res.R.cpu().numpy(), r.T) <= 1e-8
    assert _rel(res.loglik.cpu().numpy(), ll) <= 1e-8
    assert res.iterations == 5 and not res.converged


def test_pooled_loglik_under_mpc_as_numpy_shows():
    """With re-linearisation a rise is not guaranteed.  On these two simulated streams (1,000 steps, pooled, from the defaults) the
    NumPy loop of tests/em_full_oracle.py rises at every one of 10 iterations; the GPU loop is asserted to do the same."""
    _, st, z = _simulated(2, 1000, 10)
    res = kf_noise_em_full(*_args(st), z=z, iters=10, shared=True, cov_model="mpc", body_ref=st["truth"])
    pooled = res.loglik.sum(dim=1).cpu().numpy()
    print("pooled loglik", pooled)
    assert (np.diff(pooled) > 0).all()


def test_closed_loop_forces():
    """estimate_state_mpc_batch (64 trajectories x 100 steps, as in tests/test_smooth_full_gpu.py), then EM on its forces: the first
    E-step's forward pass reproduces the closed loop's x_steps bit for bit, and the loop returns finite Q, R and log-likelihoods."""
    from optistate_b200.mpc import estimate_state_mpc_batch

    T, N = 100, 64
    st = make_streams(range(N), T)
    rng = np.random.default_rng(4)
    ref = np.zeros((T, 5, 12, N))
    ref[:, :, 5, :] = 0.28
    ref[:, :, 0:3, :] = 0.02 * rng.standard_normal((T, 5, 3, N))
    xs, fs, _, _ = estimate_state_mpc_batch(st["imu"], st["p"], st["dp"], st["contact"], ref)
    body_ref = np.ascontiguousarray(ref[:, 0])
    # the first iteration of kf_noise_em_full(shared=True): the default Q / R as [12] / [10], P0 held at the starting Q
    q, r = torch.tensor(kn.Q_DEFAULT, device="cuda"), torch.tensor(kn.R_DEFAULT, device="cuda")
    first = kf_noise_stats_full(st["imu"], st["p"], st["dp"], st["contact"], fs, None, q.clone(), q, r, q_kind=nv.MAT_DIAG, r_kind=nv.MAT_DIAG,
                                p0_kind=nv.MAT_DIAG,
                                cov_model="mpc", body_ref=body_ref, n_traj=N, outputs=("x_steps",))
    assert torch.equal(first.x_steps, xs)
    em = kf_noise_em_full(st["imu"], st["p"], st["dp"], st["contact"], fs, cov_model="mpc", body_ref=body_ref, n_traj=N, shared=True,
                          iters=3)
    assert torch.equal(em.loglik[0], first.noise_stats[22])
    assert torch.isfinite(em.Q).all() and torch.isfinite(em.R).all() and torch.isfinite(em.loglik).all()
    assert int(em.status.max()) == 0
