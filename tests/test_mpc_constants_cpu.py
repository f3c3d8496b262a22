"""CPU tests of the oracle's force-MPC constants (oracle/mpc_numpy.py): the QP it builds at non-default dt, mass, inertia, gravity,
mu, fz_max and weights is still the reference's objective loop, its solver still returns KKT points there, and the defaults passed
explicitly are the module constants bit for bit (so tests/golden/mpc_reference_qp.npz pins the parametrised oracle too)."""
import numpy as np
import pytest

from oracle import mpc_numpy as mpc
from tests import mpc_cases


@pytest.mark.parametrize("name", sorted(mpc_cases.CONSTANT_SETS))
def test_condensed_qp_equals_the_objective_loop_at_other_constants(name):
    consts = mpc_cases.CONSTANT_SETS[name]
    qp_kw, _ = mpc_cases.oracle_kw(consts)
    rng = np.random.default_rng(31)
    for lateral in (0.0, 3.0):
        x, ref, p = mpc_cases.problem(rng, lateral=lateral)
        H, g, c0 = mpc.build_qp(x, ref, p, **qp_kw)
        assert np.abs(H - H.T).max() < 1e-15 * np.abs(H).max()
        assert np.linalg.eigvalsh(H).min() >= 2.0 * consts["w_force"] * (1 - 1e-9)
        for _ in range(4):
            F = 0.3 * consts["fz_max"] * rng.standard_normal((12, 5))
            u = F.T.reshape(-1)
            want = mpc.rollout_cost(F, x, ref, p, **qp_kw)
            assert abs(0.5 * u @ H @ u + g @ u + c0 - want) < 1e-10 * abs(want), (lateral, want)
    # every constant reaches the cost: changing any one of them alone changes the objective at the same forces
    x, ref, p = mpc_cases.problem(rng, lateral=0.5)
    F = 20.0 * rng.standard_normal((12, 5))
    base = mpc.rollout_cost(F, x, ref, p, **qp_kw)
    for key in qp_kw:
        other = dict(qp_kw)
        other[key] = 1.5 * np.asarray(qp_kw[key], float) + (0.1 if key == "w_state" else 0.0)
        assert abs(mpc.rollout_cost(F, x, ref, p, **other) - base) > 1e-9 * abs(base), key


@pytest.mark.parametrize("name", sorted(mpc_cases.CONSTANT_SETS))
def test_oracle_solver_returns_kkt_points_at_other_constants(name):
    consts = mpc_cases.CONSTANT_SETS[name]
    qp_kw, con_kw = mpc_cases.oracle_kw(consts)
    x, ref, p, c = mpc_cases.batch(64, seed=3)
    fz_max, mu = consts["fz_max"], consts["mu"]
    capped = friction = 0
    for k in range(64):                                  # all 16 contact patterns, each at four lateral demands
        H, g, _ = mpc.build_qp(x[:, k], ref[:, :, k].T, p[:, k], **qp_kw)
        A, b, pinned = mpc.constraints(c[:, k], **con_kw)
        assert A.shape[0] == 6 * 5 * int(c[:, k].sum()) and pinned.size == 3 * 5 * int((c[:, k] == 0).sum())
        u = mpc.solve_ldp(H, g, A, b, pinned)
        viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
        assert viol < 1e-9 * fz_max / 150.0 and stat < 1e-10, (k, c[:, k], viol, stat)
        assert np.all(u[pinned] == 0)
        F = u.reshape(5, 12)
        capped += int((np.abs(F[:, 2::3] - fz_max) < 1e-6 * fz_max).sum())
        friction += int(((np.abs(np.abs(F[:, 0::3]) - mu * F[:, 2::3]) < 1e-7 * fz_max) & (F[:, 2::3] > 1.0)).sum())
    assert capped > 0 and friction > 0, (capped, friction)  # the batch makes the fz cap and the friction pyramid bind


def test_explicit_defaults_are_the_module_constants():
    x, ref, p, c = mpc_cases.batch(16, seed=9)
    defaults = dict(mass=mpc.MASS, inertia=mpc.INERTIA, gravity=-9.81, w_state=mpc.Q_W, w_force=mpc.R_W)
    from optistate_b200.mpc import FZ_MAX, MU, W_FORCE, W_STATE
    from optistate_b200.settings import INITIAL_PARAMS

    # the oracle's defaults are the product's
    assert (mpc.MU, mpc.FZ_MAX, mpc.R_W, tuple(mpc.Q_W)) == (MU, FZ_MAX, W_FORCE, W_STATE)
    assert mpc.MASS == INITIAL_PARAMS.ROBOT_MASS and np.array_equal(mpc.INERTIA, np.diag(INITIAL_PARAMS.INERTIA_ROT))
    assert mpc.GRAV[11] == INITIAL_PARAMS.GRAVITY
    rng = np.random.default_rng(4)
    for k in range(16):
        args = (x[:, k], ref[:, :, k].T, p[:, k])
        for a, b in zip(mpc.build_qp(*args), mpc.build_qp(*args, dt=0.01, **defaults)):
            assert np.array_equal(a, b)
        for a, b in zip(mpc.constraints(c[:, k]), mpc.constraints(c[:, k], mu=0.6, fz_max=150.0)):
            assert np.array_equal(a, b)
        F = 40.0 * rng.standard_normal((12, 5))
        assert mpc.rollout_cost(F, *args) == mpc.rollout_cost(F, *args, dt=0.01, **defaults)
        assert np.array_equal(mpc.solve(*args, c[:, k]), mpc.solve(*args, c[:, k], dt=0.01, mu=0.6, fz_max=150.0, **defaults))
        A0, B0 = mpc.dynamics(args[0][0:3], args[2])
        A1, B1 = mpc.dynamics(args[0][0:3], args[2], mass=mpc.MASS, inertia=mpc.INERTIA)
        assert np.array_equal(A0, A1) and np.array_equal(B0, B1)
