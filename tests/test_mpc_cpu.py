"""CPU tests of SURVEY 8(f) row 3 (convex force MPC): the oracle restates the reference's QP consistently, its solver
returns KKT points, and the C ABI validates its descriptor.  Parity with qpOASES itself is unpinned (not available
offline; no reference fixture) - see oracle/mpc_numpy.py."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import mpc_numpy as mpc
from tests import mpc_cases


def test_condensed_qp_equals_the_reference_objective_loop():
    rng = np.random.default_rng(1)
    x, ref, p = mpc_cases.problem(rng, lateral=0.5)
    H, g, c0 = mpc.build_qp(x, ref, p)
    assert np.abs(H - H.T).max() < 1e-15 and np.linalg.eigvalsh(H).min() >= 2e-6 * (1 - 1e-9)  # strictly convex: R > 0
    for _ in range(5):
        F = 30.0 * rng.standard_normal((12, 5))
        u = F.T.reshape(-1)
        want = mpc.rollout_cost(F, x, ref, p)  # force_controller.py:70-104, literally
        assert abs(0.5 * u @ H @ u + g @ u + c0 - want) < 1e-10 * abs(want)


def test_oracle_solver_returns_kkt_points_for_every_contact_pattern():
    x, ref, p, c = mpc_cases.batch(64, seed=3)
    for k in range(64):
        H, g, _ = mpc.build_qp(x[:, k], ref[:, :, k].T, p[:, k])
        A, b, pinned = mpc.constraints(c[:, k])
        u = mpc.solve_ldp(H, g, A, b, pinned)
        viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
        assert viol < 1e-9 and stat < 1e-10, (k, c[:, k], viol, stat)
        assert np.all(u[pinned] == 0)
    # a perturbed point is NOT certified (the certificate is not vacuous)
    bad = u.copy()
    free = np.setdiff1d(np.arange(60), pinned)
    bad[free[2]] += 1e-3
    assert max(mpc.kkt_certificate(bad, H, g, A, b, pinned)) > 1e-7


P, D = ctypes.c_void_p, ctypes.c_double


class _MpcDesc(ctypes.Structure):  # OptiKfMpcDesc (include/optistate_kf.h)
    _fields_ = [("struct_size", ctypes.c_uint32), ("abi_version", ctypes.c_uint32), ("dtype", ctypes.c_int32), ("max_free_legs", ctypes.c_int32),
                ("n_problems", ctypes.c_int64), ("x", P), ("body_ref", P), ("p", P), ("contact", P), ("forces", P), ("status", P),
                ("warm_set", P), ("warm_mult", P), ("solver", ctypes.c_int32), ("max_changes", ctypes.c_int32), ("reserved0", ctypes.c_int32), ("dt", D), ("mass", D), ("inertia", D * 3), ("gravity", D), ("mu", D), ("fz_max", D), ("w_state", D * 12), ("w_force", D)]


def _mpc_lib_and_desc():
    """The library and a descriptor of four problems with valid constants and no pointers."""
    from optistate_b200 import _build

    lib = ctypes.CDLL(_build.build_all()[0])
    d = _MpcDesc(struct_size=ctypes.sizeof(_MpcDesc), abi_version=lib.optistate_kf_abi_version(), dtype=0, n_problems=4, dt=0.01, mass=8.8,
                 gravity=-9.81, mu=0.6, fz_max=150.0, w_force=1e-6)
    d.inertia = (D * 3)(0.055, 0.060, 0.105)
    d.w_state = (D * 12)(*([1.0] * 12))
    return lib, d


def test_mpc_descriptor_validation():
    lib, d = _mpc_lib_and_desc()
    assert lib.optistate_kf_mpc_forces(ctypes.byref(d), None) == -1  # pointers missing
    d.dtype = 1
    assert lib.optistate_kf_mpc_forces(ctypes.byref(d), None) == -3  # FP64 only
    d.dtype, d.mu = 0, 0.0
    assert lib.optistate_kf_mpc_forces(ctypes.byref(d), None) == -4
    d.mu, d.max_free_legs = 0.6, 5
    assert lib.optistate_kf_mpc_forces(ctypes.byref(d), None) == -4
    d.max_free_legs = 2
    d.mu, d.n_problems = 0.6, 0
    assert lib.optistate_kf_mpc_forces(ctypes.byref(d), None) == 0   # nothing to do
    d.struct_size -= 8
    assert lib.optistate_kf_mpc_forces(ctypes.byref(d), None) == -2
    assert lib.optistate_kf_mpc_forces(None, None) == -1


# Where a device is present, a descriptor that passes validation would launch kernels on the fake pointers.
@pytest.mark.skipif(torch.cuda.is_available(), reason="runs only without a CUDA device")
def test_mpc_forces_requires_a_status_array():
    """The dual active set marks the problems it hands to the interior point in `status`; without it every problem would go to
    the slower interior point, so a call without one is refused."""
    lib, d = _mpc_lib_and_desc()
    fake = ctypes.c_void_p(0x1000)  # never dereferenced: validation only
    for n in ("x", "body_ref", "p", "contact", "forces", "warm_set", "warm_mult"):
        setattr(d, n, fake)
    assert lib.optistate_kf_mpc_forces(ctypes.byref(d), None) == -1


def _oracle_verdict(f, x, ref, p, contact):
    """(cost, feasible) of forces (12, 5) by the oracle's restatement."""
    H, g, c0 = mpc.build_qp(x, ref, p)
    A, b, pinned = mpc.constraints(contact)
    u = np.asarray(f, float).T.reshape(-1)
    feasible = bool((A @ u <= b).all() if A.shape[0] else True) and bool((u[pinned] == 0).all())
    return mpc.rollout_cost(f, x, ref, p), 0.5 * u @ H @ u + g @ u + c0, feasible


def test_oracle_qp_is_the_reference_stance_controller_golden():
    """tests/golden/mpc_reference_qp.npz holds what the UNMODIFIED reference set-up code (StanceController.__init__,
    force_controller.py:44-156, run numerically through oracle/mpc_ref_shim.py) evaluates for 80 force vectors: objective
    value and whether every subject_to holds - including vectors that break exactly one constraint (fz = 150.5, |fx| =
    0.61 fz, a swing force of 1e-3) next to their just-feasible twins.  The oracle's QP is that QP."""
    import os

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mpc_reference_qp.npz"))
    assert g["cost"].shape[0] == 80 and 20 < int(g["feasible"].sum()) < 60
    for k in range(g["cost"].shape[0]):
        rollout, condensed, feasible = _oracle_verdict(g["forces"][k], g["x"][k], g["body_ref"][k], g["p"][k], g["contact"][k])
        assert abs(rollout - g["cost"][k]) <= 1e-12 * abs(g["cost"][k]), k
        assert abs(condensed - g["cost"][k]) <= 1e-10 * abs(g["cost"][k]), k
        assert feasible == bool(g["feasible"][k]), (k, g["contact"][k])


def test_oracle_qp_against_the_live_reference_set_up():
    from oracle import mpc_ref_shim as shim

    if not shim.available():
        pytest.skip("reference tree not present (GPU box)")
    rng = np.random.default_rng(11)
    for contact in ([1, 0, 0, 1], [1, 1, 1, 1], [0, 1, 0, 0]):
        x, ref, p = mpc_cases.problem(rng, lateral=0.5)
        for scale in (1.0, 40.0):
            f = scale * rng.standard_normal((12, 5))
            cost, feasible = shim.evaluate(f, x, ref, p, contact)
            rollout, condensed, ofeas = _oracle_verdict(f, x, ref, p, contact)
            assert abs(rollout - cost) <= 1e-12 * abs(cost) and abs(condensed - cost) <= 1e-10 * abs(cost) and ofeas == feasible
        # the oracle's minimiser is feasible for the reference and no feasible perturbation of it has a lower reference cost
        opt = mpc.solve(x, ref, p, contact)
        inner = np.zeros((12, 5))
        for l in range(4):
            if contact[l] == 1:
                inner[3 * l + 2] = 10.0
        c_opt, _ = shim.evaluate(opt, x, ref, p, contact)
        for _ in range(10):
            d = rng.standard_normal((12, 5)) * (np.repeat(np.asarray(contact, float), 3)[:, None] == 1)
            cand = opt + 1e-3 * (0.5 * (inner - opt) + 0.05 * d)   # moves into the interior of the feasible set
            c, feas = shim.evaluate(cand, x, ref, p, contact)
            assert feas and c >= c_opt - 1e-12 * abs(c_opt)
