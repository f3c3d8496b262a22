"""Seeded force-MPC problems shared by the CPU (oracle) and GPU tests of SURVEY 8(f) row 3."""
import numpy as np

NOMINAL_FEET = np.array([0.2, 0.15, -0.28, 0.2, -0.15, -0.28, -0.2, 0.15, -0.28, -0.2, -0.15, -0.28])


def problem(rng, lateral=0.0, height_error=False, ref_on_ground=False):
    """One problem: current state x (12), horizon reference body_ref (12, 5), body-frame feet p (12)."""
    x = np.array([0.02, -0.03, 0.1, 0, 0, 0.27, 0.1, -0.1, 0.05, 0.2, -0.1, 0.0]) + 0.01 * rng.standard_normal(12)
    ref = np.zeros((12, 5))
    ref[5] = 0.28
    ref[0:3] = 0.02 * rng.standard_normal((3, 5))
    ref[9] = lateral                                   # demanded forward velocity: large values saturate friction and fz
    ref[3] = x[3] + lateral * 0.01 * np.arange(1, 6)
    if height_error:
        x[5] = 0.1
    if ref_on_ground:
        ref[5] = 0.0
    p = NOMINAL_FEET + 0.02 * rng.standard_normal(12)
    return x, ref, p


def batch(n, seed=0):
    """n problems cycling through all 16 contact patterns and the demand / error variants; arrays in device layout
    x [12, n], body_ref [5, 12, n], p [12, n], contact [4, n]."""
    rng = np.random.default_rng(seed)
    xs, refs, ps, cs = [], [], [], []
    for k in range(n):
        contact = np.array([(k >> b) & 1 for b in range(4)], float)
        x, ref, p = problem(rng, lateral=[0.0, 0.5, 3.0, -2.0][(k // 16) % 4], height_error=k % 7 == 0, ref_on_ground=k % 11 == 0)
        xs.append(x), refs.append(ref.T), ps.append(p), cs.append(contact)
    return (np.stack(xs, axis=1), np.stack(refs, axis=2), np.stack(ps, axis=1), np.stack(cs, axis=1))


# Non-default MPC constants, as the keyword arguments of optistate_b200.mpc.mpc_forces (and of the oracle's solve).  Per-axis weights
# that differ within the position and velocity groups catch an axis mix-up in the closed-form part of H; each set has a zero weight.
HEAVY = dict(dt=0.01, mass=20.0, inertia=(0.15, 0.32, 0.41), gravity=-9.81, mu=0.4, fz_max=300.0,
             w_state=(20.0, 6.0, 0.0, 40.0, 160.0, 90.0, 2.0, 0.5, 4.0, 3.0, 0.7, 1.5), w_force=2e-6)
LIGHT = dict(dt=0.02, mass=4.5, inertia=(0.021, 0.047, 0.058), gravity=-9.81, mu=0.85, fz_max=80.0,
             w_state=(5.0, 15.0, 8.0, 250.0, 60.0, 120.0, 0.0, 2.0, 1.0, 0.4, 2.5, 6.0), w_force=1e-5)
LOW_G = dict(dt=0.005, mass=12.0, inertia=(0.071, 0.043, 0.094), gravity=-3.71, mu=0.3, fz_max=200.0,
             w_state=(12.0, 9.0, 3.0, 70.0, 20.0, 150.0, 1.5, 3.0, 0.0, 2.0, 5.0, 0.6), w_force=3e-6)
CONSTANT_SETS = {"heavy": HEAVY, "light": LIGHT, "low_g": LOW_G}


def oracle_kw(consts):
    """Splits mpc_forces-style constants into the keyword arguments of the oracle's build_qp and constraints."""
    qp = {k: consts[k] for k in ("dt", "mass", "inertia", "gravity", "w_state", "w_force") if k in consts}
    con = {k: consts[k] for k in ("mu", "fz_max") if k in consts}
    return qp, con
