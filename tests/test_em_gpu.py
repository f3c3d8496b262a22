"""GPU tests of the EM E-step (kf_noise_stats) and the EM loop (kf_noise_em): the CUDA statistics against the NumPy oracle of
tests/em_oracle.py, the forward and smoothed outputs against kf_batch / kf_smooth, degenerate sizes, status and refusals."""
import numpy as np
import pytest
import torch

from oracle import cases
from oracle import kf_numpy as kn
from optistate_b200 import kf_batch, kf_noise_em, kf_noise_stats, kf_smooth
from optistate_b200.batch import kf_measure
from optistate_b200.synth import make_streams, monte_carlo_noise
from tests import em_oracle as eo
from tests.test_smooth_gpu import _forward_cases

pytestmark = pytest.mark.gpu


def _streams(S, T, seed0):
    return make_streams(range(seed0, seed0 + S), T)


def _args(st):
    return st["imu"], st["p"], st["dp"], st["contact"], st["f"]


def _oracle_stats(st, kw, n):
    out = np.empty((23, n))
    P0 = kw["Q"] if kw["P0"] is None else kw["P0"]
    for j in range(n):
        s = {k: v[:, :, j] for k, v in st.items()}
        Sw, Sv, ll = eo.estep_textbook(eo.forward(s, kw["x0"], P0, kw["Q"], kw["R"]), kw["Q"], kw["R"])
        out[:12, j], out[12:22, j], out[22, j] = Sw, Sv, ll
    return out


def _rel(a, b):
    return float((np.abs(a - b) / np.abs(b)).max())


@pytest.mark.parametrize("name", ["default_seed11_10k", "stress_qrpkl_seed3_10k"])
def test_fp64_matches_numpy_estep(name):
    """3 streams x 10,000 steps, FP64: every Sw / Sv row and the log-likelihood within 1e-9 relative of the NumPy oracle."""
    _, kw, _ = cases.build(name)
    st = _streams(3, 10000, 11)
    res = kf_noise_stats(*_args(st), x0=kw["x0"], Q=kw["Q"], R=kw["R"])
    got = res.noise_stats.cpu().numpy()
    ref = _oracle_stats(st, kw, 3)
    e = _rel(got, ref)
    print(f"{name}: worst relative error {e:.2e}")
    assert e <= 1e-9
    assert int(res.status.max()) == 0


def test_fp32_within_stated_tolerance():
    """FP32, default noise, 10,000 steps on two streams.  Bounds: Sw / Sv rows 2e-2 relative, log-likelihood 1e-3 relative."""
    _, kw, _ = cases.build("default_seed11_10k")
    st = _streams(2, 10000, 11)
    res = kf_noise_stats(*_args(st), x0=kw["x0"], Q=kw["Q"], R=kw["R"], dtype=torch.float32)
    got = res.noise_stats.cpu().numpy().astype(np.float64)
    ref = _oracle_stats(st, kw, 2)
    es, el = _rel(got[:22], ref[:22]), _rel(got[22], ref[22])
    print(f"fp32: stats {es:.2e}, loglik {el:.2e}")
    assert es <= 2e-2 and el <= 1e-3


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_smoothed_outputs_are_kf_smooth(dtype):
    st = _streams(64, 150, 900)
    a = kf_smooth(*_args(st), dtype=dtype, outputs=("x_smooth", "var_smooth"))
    b = kf_noise_stats(*_args(st), dtype=dtype, outputs=("x_smooth", "var_smooth"))
    assert torch.equal(a.x_smooth, b.x_smooth) and torch.equal(a.var_smooth, b.var_smooth)
    assert torch.isfinite(b.noise_stats).all()


@pytest.mark.parametrize("case", range(5))
def test_forward_pass_is_kf_batch(case):
    name, st, kw = _forward_cases()[case]
    outs = ("x_steps", "summary")
    a = kf_batch(*_args(st), outputs=outs, truth=st["truth"], **kw)
    b = kf_noise_stats(*_args(st), outputs=outs, truth=st["truth"], **kw)
    assert b.algo == "sequential", name
    for o in outs:
        assert torch.equal(a.tensors[o], b.tensors[o]), (name, o)
    assert torch.equal(a.status, b.status), name
    assert torch.isfinite(b.noise_stats).all(), name


def test_streamed_and_direct_paths_agree_and_caller_z():
    name, st, kw = _forward_cases()[0]
    _, _, kwd = _forward_cases()[1]
    a = kf_noise_stats(*_args(st), **kw)
    b = kf_noise_stats(*_args(st), **kwd)
    assert torch.equal(a.noise_stats, b.noise_stats)
    z, _ = kf_measure(st["imu"], st["p"], st["dp"], st["contact"])
    c = kf_noise_stats(None, st["p"], None, None, st["f"], z=z, **kw)
    assert torch.equal(a.noise_stats, c.noise_stats)


def test_degenerate_sizes():
    st = _streams(8, 30, 950)
    one = {k: v[:1] for k, v in st.items()}
    r1 = kf_noise_stats(*_args(one))  # T = 1: the t = -1 transition and the first measurement only
    kw = dict(x0=None, P0=None, Q=np.diag(kn.Q_DEFAULT), R=np.diag(kn.R_DEFAULT))
    assert _rel(r1.noise_stats.cpu().numpy(), _oracle_stats(one, kw, 8)) <= 1e-9
    r0 = kf_noise_stats(*_args({k: v[:0] for k, v in st.items()}))
    assert r0.noise_stats.shape == (23, 8) and not r0.noise_stats.any()
    rn = kf_noise_stats(*_args(st), n_traj=0, outputs=("x_smooth",))
    assert rn.noise_stats.shape == (23, 0) and rn.x_smooth.shape == (30, 12, 0)


def test_singular_prior_sets_smooth_not_pd():
    st = _streams(32, 50, 700)
    q = np.diag(cases.Q_DEFAULT).copy()
    q[[3, 9]] = 0.0
    res = kf_noise_stats(*_args(st), Q=q, P0=q)
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
            kf_noise_stats(*_args(st), **kw)


Q_TRUE, R_TRUE = kn.Q_DEFAULT * 0.5, kn.R_DEFAULT * 2.0


def _simulated(S, T, seed0=0):
    sims = [eo.simulate(seed0 + j, T, Q_TRUE, R_TRUE) for j in range(S)]
    st = {k: np.ascontiguousarray(np.stack([s[0][k] for s in sims], axis=-1)) for k in sims[0][0]}
    z = np.ascontiguousarray(np.stack([s[1] for s in sims], axis=-1))
    return sims, st, z


def test_em_matches_numpy_shared_and_per_member():
    """5 iterations on 4 simulated streams: Q, R and the log-likelihood equal the NumPy EM loop to 1e-8 relative, pooled, and
    per trajectory for Monte-Carlo members that share the streams and start from different Q / R."""
    sims, st, z = _simulated(4, 200)
    res = kf_noise_em(st["imu"], st["p"], st["dp"], st["contact"], st["f"], z=z, iters=5, shared=True)
    q, r, ll = eo.em([s[0] for s in sims], kn.Q_DEFAULT, kn.R_DEFAULT, 5, True, zs=[s[1] for s in sims])
    assert _rel(res.Q.cpu().numpy(), q) <= 1e-8 and _rel(res.R.cpu().numpy(), r) <= 1e-8
    assert _rel(res.loglik.cpu().numpy(), ll) <= 1e-8
    pooled = res.loglik.sum(dim=1).cpu().numpy()
    assert (np.diff(pooled) >= 0).all(), pooled
    N = 8
    q0, r0 = monte_carlo_noise(np.arange(N), kn.Q_DEFAULT, kn.R_DEFAULT)
    idx = (np.arange(N) % 4).astype(np.int32)
    res = kf_noise_em(st["imu"], st["p"], st["dp"], st["contact"], st["f"], Q=q0, R=r0, z=z, iters=5, n_traj=N, stream_index=idx)
    q, r, ll = eo.em([sims[j][0] for j in idx], q0.T, r0.T, 5, False, zs=[sims[j][1] for j in idx])
    assert _rel(res.Q.cpu().numpy(), q.T) <= 1e-8 and _rel(res.R.cpu().numpy(), r.T) <= 1e-8
    assert _rel(res.loglik.cpu().numpy(), ll) <= 1e-8
    assert res.iterations == 5 and not res.converged


def test_pooled_loglik_rises_and_tol_stops():
    _, st, z = _simulated(2, 1000, 10)
    res = kf_noise_em(st["imu"], st["p"], st["dp"], st["contact"], st["f"], z=z, iters=14, shared=True)
    pooled = res.loglik.sum(dim=1).cpu().numpy()
    print("pooled loglik", pooled)
    assert (np.diff(pooled) > 0).all()
    res2 = kf_noise_em(st["imu"], st["p"], st["dp"], st["contact"], st["f"], z=z, iters=50, tol=1e-3, shared=True)
    assert res2.converged and res2.iterations < 50


def test_recovery_of_simulated_noise():
    """256 streams x 1,000 steps simulated with Q = 0.5 Q_default, R = 2 R_default; pooled EM from the defaults, 40 iterations.
    The components the model identifies come within 10 % of the truth (DESIGN.md section 0 lists those that do not)."""
    _, st, z = _simulated(256, 1000, 1000)
    res = kf_noise_em(st["imu"], st["p"], st["dp"], st["contact"], st["f"], z=z, iters=40, shared=True)
    qr = res.Q.cpu().numpy() / Q_TRUE
    rr = res.R.cpu().numpy() / R_TRUE
    print("q / q_true", np.round(qr, 3), "r / r_true", np.round(rr, 3))
    assert (np.abs(qr[[0, 1, 2, 5, 9, 10]] - 1) <= 0.1).all()
    assert (np.abs(rr[[0, 1, 2, 3, 7, 8, 9]] - 1) <= 0.1).all()
