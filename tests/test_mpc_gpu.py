"""GPU tests of SURVEY 8(f) row 3: the batched force MPC (csrc/kf_mpc.cuh, one warp per QP) against the oracle's
independent active-set solve and a solver-independent KKT certificate.  Parity with qpOASES is unpinned (see
oracle/mpc_numpy.py); the QP is strictly convex, so agreement with any exact solver is agreement with the minimiser."""
import numpy as np
import pytest
import torch

from optistate_b200 import Kalman_Filter
from optistate_b200.mpc import ST_UNPOLISHED, mpc_forces
from oracle import mpc_numpy as mpc
from tests import mpc_cases

pytestmark = pytest.mark.gpu


def test_forces_are_the_minimiser_for_all_contact_patterns_and_saturations():
    n = 256
    x, ref, p, c = mpc_cases.batch(n, seed=0)
    forces, status = mpc_forces(x, ref, p, c)
    torch.cuda.synchronize()
    F, st = forces.cpu().numpy(), status.cpu().numpy()
    assert F.shape == (5, 12, n)
    assert not (st & ST_UNPOLISHED).any(), np.where(st & ST_UNPOLISHED)[0]
    worst = 0.0
    for k in range(n):
        H, g, _ = mpc.build_qp(x[:, k], ref[:, :, k].T, p[:, k])
        A, b, pinned = mpc.constraints(c[:, k])
        u = F[:, :, k].reshape(-1)
        viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
        assert viol < 1e-7 and stat < 1e-8, (k, c[:, k], viol, stat)            # feasible to 1e-7 N, stationary to 1e-8 |g|
        want = mpc.solve_ldp(H, g, A, b, pinned)
        err = np.abs(u - want).max() / max(1.0, np.abs(want).max())
        worst = max(worst, err)
        assert err < 1e-8, (k, c[:, k], err)
        assert np.all(u[pinned] == 0.0)
    print("worst |u - u_oracle| / max|u|:", worst, " interior-point iterations max:", int((st >> 8).max()))
    # saturation really occurs in the batch: friction faces and the fz cap
    assert (np.abs(F[:, 2::3, :] - 150.0) < 1e-6).any() and (np.abs(np.abs(F[:, 0::3, :]) - 0.6 * F[:, 2::3, :]) < 1e-7)[F[:, 2::3, :] > 1].any()


def test_all_swing_and_unconstrained_legs():
    x, ref, p, c = mpc_cases.batch(16, seed=5)
    c[:] = 0.0
    forces, status = mpc_forces(x, ref, p, c)
    assert torch.count_nonzero(forces) == 0 and not (status & 3).any()
    # a contact value that is neither 0 nor 1 leaves the leg unconstrained (the reference's if_else selects neither set)
    c[:] = 0.5
    forces, status = mpc_forces(x, ref, p, c)
    F = forces.cpu().numpy()
    for k in range(4):
        H, g, _ = mpc.build_qp(x[:, k], ref[:, :, k].T, p[:, k])
        want = np.linalg.solve(H, -g)
        assert np.abs(F[:, :, k].reshape(-1) - want).max() < 1e-8 * max(1.0, np.abs(want).max())


def test_estimate_state_mpc_solves_for_its_forces_on_the_device():
    """The drop-in class without a force provider: predict_mpc solves the reference's QP (kalman_filter.py:147-152)."""
    rng = np.random.default_rng(2)
    x, ref, p = mpc_cases.problem(rng, lateral=0.5)
    contact = np.array([1.0, 0.0, 0.0, 1.0]).reshape(4, 1)
    kf = Kalman_Filter()
    kf.x = x.reshape(12, 1).copy()
    imu = np.concatenate([x[0:3], x[6:9]]).reshape(6, 1)
    dp = 0.05 * rng.standard_normal((12, 1))
    p_in = p.reshape(12, 1).copy()
    kf.estimate_state_mpc(imu, p_in, dp, ref, contact)
    want = mpc.solve(x, ref, p, contact)            # (12, 5)
    assert kf.f.shape == (12, 5)
    assert np.abs(kf.f - want).max() < 1e-8 * np.abs(want).max()
    # same step with the oracle's forces supplied explicitly gives the same state
    kf2 = Kalman_Filter()
    kf2.x = x.reshape(12, 1).copy()
    kf2.estimate_state_mpc(imu, p.reshape(12, 1).copy(), dp, ref, contact, f=want)
    assert np.abs(kf.x - kf2.x).max() < 1e-10


def test_batched_closed_loop_equals_the_class_loop():
    """estimate_state_mpc_batch (MPC from the current estimate + one filter step, per step, for all trajectories) against the
    drop-in class driven trajectory by trajectory."""
    from optistate_b200.mpc import estimate_state_mpc_batch
    from optistate_b200.synth import make_streams

    T, N = 6, 3
    st = make_streams(range(N), T)
    rng = np.random.default_rng(4)
    ref = np.zeros((T, 5, 12, N))
    ref[:, :, 5, :] = 0.28
    ref[:, :, 0:3, :] = 0.02 * rng.standard_normal((T, 5, 3, N))
    xs, fs, mst, fst = estimate_state_mpc_batch(st["imu"], st["p"], st["dp"], st["contact"], ref)
    torch.cuda.synchronize()
    assert not (mst & ST_UNPOLISHED).any() and int(fst.max()) == 0
    for n in range(N):
        kf = Kalman_Filter()
        kf.x = kf.x.copy()
        for t in range(T):
            x = kf.estimate_state_mpc(st["imu"][t, :, n].reshape(6, 1), st["p"][t, :, n].reshape(12, 1).copy(), st["dp"][t, :, n].reshape(12, 1),
                                      ref[t, :, :, n].T, st["contact"][t, :, n].reshape(4, 1))
            assert np.abs(kf.f[:, 0] - fs[t, :, n].cpu().numpy()).max() < 1e-6 * max(1.0, np.abs(kf.f[:, 0]).max()), (n, t)
            assert np.abs(x.reshape(12) - xs[t, :, n].cpu().numpy()).max() < 1e-7, (n, t)


def test_shared_memory_bound_on_the_legs_out_of_swing():
    """max_free_legs sizes the kernel's shared memory: same forces with the tight bound, a flagged NaN when it is wrong."""
    from optistate_b200.mpc import ST_TOO_MANY_LEGS

    x, ref, p, c = mpc_cases.batch(64, seed=7)
    c[:] = np.array([1.0, 0.0, 0.0, 1.0])[:, None]  # a trot: two legs in stance
    loose, _ = mpc_forces(x, ref, p, c, max_free_legs=4)   # the shared-memory kernel (kf_mpc.cuh)
    tight, st = mpc_forces(x, ref, p, c)              # bound taken from the contact array: 2 - the one-warp kernel (kf_mpc_gi.cuh)
    assert float((loose - tight).abs().max()) < 1e-8 * float(tight.abs().max()) and not (st & 7).any()
    c[:, 5] = 1.0                                      # one problem with four legs in stance, but the caller promises two
    wrong, st = mpc_forces(x, ref, p, c, max_free_legs=2)
    assert int(st[5]) == ST_TOO_MANY_LEGS and torch.isnan(wrong[:, :, 5]).all()
    keep = torch.arange(64) != 5
    assert torch.equal(wrong[:, :, keep], tight[:, :, keep])


def test_trot_batch_polishes_every_problem():
    """4,096 trot problems; number 833 made simultaneous active-set corrections cycle (period 4) until the corrections were
    limited to one change per round after the second round."""
    x, ref, p, c = mpc_cases.batch(4096, seed=1)
    c[:] = np.where((np.arange(4096) % 2 == 0)[None, :], np.array([1.0, 0, 0, 1])[:, None], np.array([0, 1.0, 1, 0])[:, None])
    forces, status = mpc_forces(x, ref, p, c)
    F, st = forces.cpu().numpy(), status.cpu().numpy()
    assert not (st & 7).any(), np.where(st & 7)[0]
    for k in [833] + list(range(0, 4096, 128)):
        H, g, _ = mpc.build_qp(x[:, k], ref[:, :, k].T, p[:, k])
        A, b, pinned = mpc.constraints(c[:, k])
        want = mpc.solve_ldp(H, g, A, b, pinned)
        u = F[:, :, k].reshape(-1)
        assert np.abs(u - want).max() < 1e-8 * max(1.0, np.abs(want).max()), k
        viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
        assert viol < 1e-7 and stat < 1e-8, (k, viol, stat)


def test_dual_active_set_warm_start_and_solver_agreement():
    """The default solver for a trot (kf_mpc_gi.cuh) against the interior-point kernel on the same problems, and its warm start: the
    working set of one solve, entered by bordering, starts the next one - same minimiser, fewer iterations, also when the set has
    to change or belongs to other legs."""
    from optistate_b200.mpc import ST_WARM, WarmStart

    n = 1024
    x, ref, p, c = mpc_cases.batch(n, seed=11)
    c[:] = np.where((np.arange(n) % 2 == 0)[None, :], np.array([1.0, 0, 0, 1])[:, None], np.array([0, 1.0, 1, 0])[:, None])
    c[:, ::17] = np.array([0.0, 1.0, 0.0, 0.0])[:, None]          # a few problems with a single stance leg
    gi, st = mpc_forces(x, ref, p, c)
    ipm, st_ip = mpc_forces(x, ref, p, c, solver="interior_point")
    scale = float(ipm.abs().max())
    assert not (st & 7).any() and not (st_ip & 7).any()
    assert float((gi - ipm).abs().max()) < 1e-8 * scale
    warm = WarmStart(n)
    first, s0 = mpc_forces(x, ref, p, c, warm=warm)
    assert torch.equal(first, gi) and not (s0 & ST_WARM).any()
    again, s1 = mpc_forces(x, ref, p, c, warm=warm)               # same problems: the set is the answer, no constraint enters or leaves
    constrained = (warm.active[0] & 0xFFFFF) != 0
    assert float((again - gi).abs().max()) < 1e-9 * scale and bool(((s1 & ST_WARM) != 0)[constrained].all())
    assert int((s1 >> 8)[constrained].max()) == 0
    rng = np.random.default_rng(5)
    x2 = x + 2e-3 * rng.standard_normal(x.shape)
    ref2 = ref + 1e-3 * rng.standard_normal(ref.shape)
    near, s2 = mpc_forces(x2, ref2, p, c, warm=warm)
    plain, s2c = mpc_forces(x2, ref2, p, c)
    assert not (s2 & 7).any() and float((near - plain).abs().max()) < 1e-8 * scale
    assert float((s2 >> 8).double().mean()) < 0.5 * float((s2c >> 8).double().mean())   # far fewer constraint changes than from scratch
    c2 = 1.0 - c
    c2[:, ::17] = np.array([0.0, 0.0, 1.0, 0.0])[:, None]
    sw, s3 = mpc_forces(x2, ref2, p, c2, warm=warm)
    sw_cold, _ = mpc_forces(x2, ref2, p, c2)
    assert not (s3 & (7 | ST_WARM)).any() and torch.equal(sw, sw_cold)
    F = near.cpu().numpy()
    for k in list(range(0, n, 61)) + [0, 17, 34]:
        H, g, _ = mpc.build_qp(x2[:, k], ref2[:, :, k].T, p[:, k])
        A, b, pinned = mpc.constraints(c[:, k])
        want = mpc.solve_ldp(H, g, A, b, pinned)
        u = F[:, :, k].reshape(-1)
        assert np.abs(u - want).max() < 1e-8 * max(1.0, np.abs(want).max()), k
        viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
        assert viol < 1e-7 and stat < 1e-8, (k, viol, stat)


def test_dual_active_set_with_two_warps_covers_three_and_four_stance_legs():
    """Orders 45 and 60 (three and four legs out of swing) run the same dual active-set method with two warps per problem
    (kf_mpc_gi2_kernel); a mixed batch exercises every instantiation, the shared-memory interior point (kf_mpc.cuh) is the yardstick,
    and a standing batch (all four legs in stance) carries a warm start from one solve to the next."""
    from optistate_b200.mpc import ST_WARM, WarmStart

    n = 512
    x, ref, p, c = mpc_cases.batch(n, seed=21)
    gi, st = mpc_forces(x, ref, p, c)
    ipm, st_ip = mpc_forces(x, ref, p, c, solver="interior_point")
    scale = float(ipm.abs().max())
    assert not (st & 7).any() and not (st_ip & 7).any()
    assert float((gi - ipm).abs().max()) < 1e-8 * scale
    four = np.ones((4, n))
    stand, s0 = mpc_forces(x, ref, p, four)
    stand_ip, _ = mpc_forces(x, ref, p, four, solver="interior_point")
    assert not (s0 & 7).any() and float((stand - stand_ip).abs().max()) < 1e-8 * float(stand_ip.abs().max())
    F = stand.cpu().numpy()
    for k in range(0, n, 41):
        H, g, _ = mpc.build_qp(x[:, k], ref[:, :, k].T, p[:, k])
        A, b, pinned = mpc.constraints(four[:, k])
        want = mpc.solve_ldp(H, g, A, b, pinned)
        u = F[:, :, k].reshape(-1)
        assert np.abs(u - want).max() < 1e-8 * max(1.0, np.abs(want).max()), k
        viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
        assert viol < 1e-7 and stat < 1e-8, (k, viol, stat)
    warm = WarmStart(n)
    mpc_forces(x, ref, p, four, warm=warm)
    again, s1 = mpc_forces(x, ref, p, four, warm=warm)
    constrained = (warm.active[0] & 0xFFFFF) != 0
    assert float((again - stand).abs().max()) < 1e-9 * float(stand.abs().max()) and bool(((s1 & ST_WARM) != 0)[constrained].all())
    assert int((s1 >> 8)[constrained].max()) == 0


def test_batched_closed_loop_with_dense_noise_custom_p0_and_dt():
    """Non-default arguments of estimate_state_mpc_batch: a dense Q (joint filter step, like the class), a per-call P0, another dt -
    the model constants reach the MPC AND the filter - against the drop-in class driven step by step."""
    from optistate_b200.mpc import estimate_state_mpc_batch
    from optistate_b200.synth import make_streams

    T, N = 5, 2
    st = make_streams(range(20, 20 + N), T)
    rng = np.random.default_rng(8)
    ref = np.zeros((T, 5, 12, N))
    ref[:, :, 5, :] = 0.28
    m = 0.01 * rng.standard_normal((12, 12))
    Q = np.diag(np.full(12, 0.01)) + m @ m.T                       # dense, symmetric positive definite
    R = np.diag(np.linspace(0.005, 0.02, 10))
    P0 = np.diag(np.linspace(0.01, 0.03, 12))
    dt = 0.02
    xs, fs, mst, fst = estimate_state_mpc_batch(st["imu"], st["p"], st["dp"], st["contact"], ref, P0=P0, Q=Q, R=R, dt=dt)
    torch.cuda.synchronize()
    assert not (mst & 7).any() and int((fst & 2).max()) == 0
    for n in range(N):
        kf = Kalman_Filter()
        kf.x = kf.x.copy()
        kf.Q, kf.R, kf.P, kf.dt = Q.copy(), R.copy(), P0.copy(), dt
        for t in range(T):
            x = kf.estimate_state_mpc(st["imu"][t, :, n].reshape(6, 1), st["p"][t, :, n].reshape(12, 1).copy(), st["dp"][t, :, n].reshape(12, 1),
                                      ref[t, :, :, n].T, st["contact"][t, :, n].reshape(4, 1))
            assert np.abs(kf.f[:, 0] - fs[t, :, n].cpu().numpy()).max() < 1e-6 * max(1.0, np.abs(kf.f[:, 0]).max()), (n, t)
            assert np.abs(x.reshape(12) - xs[t, :, n].cpu().numpy()).max() < 1e-7, (n, t)


def test_problems_the_dual_active_set_gives_up_on_are_solved_by_the_interior_point():
    """The hand-over path: with a budget of three constraint changes most saturated problems are flagged by the dual active-set
    kernel and solved by the interior-point kernel in the second launch - same forces as without the budget, no flag left."""
    n = 256
    x, ref, p, c = mpc_cases.batch(n, seed=13)
    for contact in (np.where((np.arange(n) % 2 == 0)[None, :], np.array([1.0, 0, 0, 1])[:, None], np.array([0, 1.0, 1, 0])[:, None]), c):
        full, st = mpc_forces(x, ref, p, contact)
        capped, st_c = mpc_forces(x, ref, p, contact, max_changes=3)
        assert not (st & 7).any() and not (st_c & (7 | 16)).any()
        took_ipm = ((st >> 8) > 3)                       # these needed more than the budget: the second launch solved them
        assert int(took_ipm.sum()) > n // 8
        assert float((capped - full).abs().max()) < 1e-8 * float(full.abs().max())
