"""TEST INFRASTRUCTURE ONLY (oracle for SURVEY 8(f) row 3) - never imported by the product package.

NumPy restatement of the reference's convex force MPC, /root/reference/misc/force_controller.py:15-225, as
`Kalman_Filter.predict_mpc` sets it up (/root/reference/kalman_filter/kalman_filter.py:64-77,140-152):

    horizon N = 5, Q = diag(10,10,10,100,100,100,1,1,5,1,1,1), R = 1e-6 I, P = Q, dt = 0.01, mu = 0.6, 0 <= fz <= 150
    body_mpc[:,0] = x, body_mpc[:,1:] = body_ref (12 x 5);  p_mpc[:, i] = p for every stage;  contact_mpc[:, i] = contact
    state_{i+1} = (I + A_i dt) state_i + B_i dt u_i + dt g        (A_i, B_i from body_mpc[:, i], p_mpc[:, i])   :70-93
    cost = sum_i (state_{i+1} - body_mpc[:, i+1])^T W_i (.) + u_i^T R u_i,  W_i = Q (i < N-1), P (i = N-1)      :95-104
    swing leg (contact == 0): f = 0;  stance leg (contact == 1): 0 <= fz <= 150, |fx| <= mu fz, |fy| <= mu fz    :106-156

PARITY: the QP is PINNED to the reference, its SOLVER is unpinned.  The reference solves this QP with CasADi 3.6.2 +
qpOASES (environment.yml:25), neither of which is available offline, and no reference test or fixture holds a force
vector.  What anchors this file:
  * oracle/mpc_ref_shim.py runs the UNMODIFIED StanceController.__init__ under a numeric stand-in for casadi, which makes
    the reference's own code evaluate its objective and its subject_to constraints for given forces;
    tests/golden/mpc_reference_qp.npz (oracle/gen_golden_mpc.py) holds 80 such evaluations, and `rollout_cost` / `build_qp` /
    `constraints` below reproduce every one of them (cost to 1e-12, feasibility verdicts exactly, including forces that
    break exactly one constraint);
  * the QP is strictly convex (R > 0), so its minimiser is unique: any correct solver returns qpOASES' answer up to solver
    tolerance.  `solve_ldp` (least-distance programming through NNLS, an active-set method - a different algorithm from
    the GPU's interior-point method) and `kkt_certificate` (solver-independent optimality check) are the checkers.
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import nnls

NH = 5
MU = 0.6
FZ_MAX = 150.0
Q_W = np.array([10.0, 10.0, 10.0, 100.0, 100.0, 100.0, 1.0, 1.0, 5.0, 1.0, 1.0, 1.0])  # kalman_filter.py:64
R_W = 1e-6                                                                               # kalman_filter.py:66
MASS = 8.8
INERTIA = np.array([55303643.08, 60119440.34, 105304340.05]) / 1e9                       # force_controller.py:32-35
GRAV = np.array([0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, -9.81])                                # force_controller.py:28


def rot_zyx(thx, thy, thz):
    """force_controller.py:168-177."""
    cx, sx, cy, sy, cz, sz = np.cos(thx), np.sin(thx), np.cos(thy), np.sin(thy), np.cos(thz), np.sin(thz)
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    return Rz @ (Ry @ Rx)


def skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])


def dynamics(th, p, *, mass=MASS, inertia=INERTIA):
    """A (force_controller.py:179-192) and B (:194-224) for reference angles th (3) and body-frame feet p (12)."""
    R = rot_zyx(*th)
    A = np.zeros((12, 12))
    A[0:3, 6:9] = R.T
    A[3:6, 9:12] = np.eye(3)
    I_hat_inv = np.linalg.inv(R @ np.diag(np.asarray(inertia, float)) @ R.T)
    B = np.zeros((12, 12))
    for leg in range(4):
        B[6:9, 3 * leg:3 * leg + 3] = I_hat_inv @ skew(R @ p[3 * leg:3 * leg + 3])
        B[9:12, 3 * leg:3 * leg + 3] = np.eye(3) / mass
    return A, B


def horizon(x, body_ref, p):
    """body_mpc (12 x 6) and p_mpc (12 x 6) as predict_mpc fills them (kalman_filter.py:141-146)."""
    body = np.concatenate([np.asarray(x, float).reshape(12, 1), np.asarray(body_ref, float).reshape(12, NH)], axis=1)
    feet = np.repeat(np.asarray(p, float).reshape(12, 1), NH + 1, axis=1)
    return body, feet


def _grav(gravity):
    """The gravity vector of the dynamics: `gravity` on the z velocity (force_controller.py:28)."""
    g = np.zeros(12)
    g[11] = gravity
    return g


def rollout_cost(u, x, body_ref, p, dt=0.01, *, mass=MASS, inertia=INERTIA, gravity=GRAV[11], w_state=Q_W, w_force=R_W):
    """The reference's objective loop, literally (force_controller.py:70-104).  u: (12, NH) forces per stage."""
    body, feet = horizon(x, body_ref, p)
    u = np.asarray(u, float).reshape(12, NH)
    w = np.asarray(w_state, float)
    Q, R, P = np.diag(w), w_force * np.eye(12), np.diag(w)
    grav = _grav(gravity)
    state, cost = body[:, 0].copy(), 0.0
    for i in range(NH):
        A, B = dynamics(body[0:3, i], feet[:, i], mass=mass, inertia=inertia)
        state = (np.eye(12) + A * dt) @ state + (B * dt) @ u[:, i] + dt * grav
        e = state - body[:, i + 1]
        cost += e @ (P if i == NH - 1 else Q) @ e + u[:, i] @ R @ u[:, i]
    return cost


def build_qp(x, body_ref, p, dt=0.01, *, mass=MASS, inertia=INERTIA, gravity=GRAV[11], w_state=Q_W, w_force=R_W):
    """Condensed form: cost(u) = 1/2 u^T H u + g^T u + c0 with u = vec of the (12, NH) forces, stage-major (u[12 i + k])."""
    body, feet = horizon(x, body_ref, p)
    n = 12 * NH
    Su, sc = np.zeros((12, n)), body[:, 0].copy()
    H, g, c0 = 2.0 * w_force * np.eye(n), np.zeros(n), 0.0
    grav = _grav(gravity)
    for i in range(NH):
        A, B = dynamics(body[0:3, i], feet[:, i], mass=mass, inertia=inertia)
        Ad = np.eye(12) + A * dt
        Su = Ad @ Su
        Su[:, 12 * i:12 * i + 12] += B * dt
        sc = Ad @ sc + dt * grav
        W = np.diag(np.asarray(w_state, float))  # P = Q
        e = sc - body[:, i + 1]
        H += 2.0 * Su.T @ W @ Su
        g += 2.0 * Su.T @ W @ e
        c0 += e @ W @ e
    return H, g, c0


def constraints(contact, *, mu=MU, fz_max=FZ_MAX):
    """A u <= b rows (and the index set of variables pinned to zero) for the contact pattern of all NH stages.
    contact == 0: f = 0 (force_controller.py:110-123);  contact == 1: friction pyramid + 0 <= fz <= fz_max (:125-156);
    any other value: the reference's if_else selects neither, the leg is unconstrained."""
    contact = np.asarray(contact, float).reshape(4)
    rows, rhs, pinned = [], [], []
    for i in range(NH):
        for leg in range(4):
            k = 12 * i + 3 * leg
            if contact[leg] == 0:
                pinned += [k, k + 1, k + 2]
            elif contact[leg] == 1:
                for coef, b in (((0, 0, -1.0), 0.0), ((0, 0, 1.0), fz_max), ((1.0, 0, -mu), 0.0), ((-1.0, 0, -mu), 0.0),
                                ((0, 1.0, -mu), 0.0), ((0, -1.0, -mu), 0.0)):
                    r = np.zeros(12 * NH)
                    r[k:k + 3] = coef
                    rows.append(r)
                    rhs.append(b)
    A = np.array(rows).reshape(-1, 12 * NH)
    return A, np.array(rhs), np.array(pinned, dtype=int)


def solve_ldp(H, g, A, b, pinned):
    """Minimiser of 1/2 u^T H u + g^T u s.t. A u <= b, pinned variables = 0, by Lawson & Hanson's least-distance
    programming: with H = L L^T and z = L^T u + L^-1 g the problem is min |z| s.t. G z >= h, which is one NNLS solve
    (scipy's Lawson-Hanson active-set code - a different algorithm from the GPU's interior-point method, and robust at
    the degenerate apex of the friction pyramid where four faces meet in three dimensions)."""
    n = H.shape[0]
    free = np.setdiff1d(np.arange(n), pinned)
    u = np.zeros(n)
    if free.size == 0:
        return u
    Hf, gf = H[np.ix_(free, free)], g[free]
    L = np.linalg.cholesky(Hf)
    d = np.linalg.solve(L, gf)
    if A.shape[0] == 0:
        u[free] = np.linalg.solve(L.T, -d)
        return u
    Af = A[:, free]
    G = -np.linalg.solve(L, Af.T).T              # -A L^-T
    h = -b - Af @ np.linalg.solve(L.T, d)        # A u <= b  <=>  G z >= h  with  u = L^-T (z - d)
    # scale rows: NNLS is scale-sensitive in its tolerances
    sc = np.maximum(np.linalg.norm(G, axis=1), 1e-300)
    G, h = G / sc[:, None], h / sc
    E = np.vstack([G.T, h[None, :]])
    f = np.zeros(free.size + 1)
    f[-1] = 1.0
    w, _ = nnls(E, f, maxiter=50 * E.shape[1])
    r = E @ w - f
    if abs(r[-1]) < 1e-300:
        raise ValueError("infeasible constraints")
    z = -r[:-1] / r[-1]
    u[free] = np.linalg.solve(L.T, z - d)
    return u


def kkt_certificate(u, H, g, A, b, pinned, act_tol=1e-7):
    """Solver-independent optimality check of a candidate u: (max constraint violation, stationarity residual relative to
    |g|) where the multipliers of the (nearly) active constraints are the best non-negative ones (NNLS)."""
    u = np.asarray(u, float).reshape(-1)
    free = np.setdiff1d(np.arange(H.shape[0]), pinned)
    viol = max(float(np.max(A @ u - b)) if A.shape[0] else 0.0, float(np.abs(u[pinned]).max()) if pinned.size else 0.0, 0.0)
    if free.size == 0:
        return viol, 0.0
    grad = (H @ u + g)[free]
    scale = max(np.abs(g[free]).max(), 1e-30)
    act = np.where(A @ u - b >= -act_tol * np.maximum(1.0, np.abs(b)))[0] if A.shape[0] else np.array([], int)
    if act.size == 0:
        return viol, float(np.abs(grad).max() / scale)
    lam, _ = nnls(A[np.ix_(act, free)].T, -grad)
    return viol, float(np.abs(grad + A[np.ix_(act, free)].T @ lam).max() / scale)


def solve(x, body_ref, p, contact, dt=0.01, *, mass=MASS, inertia=INERTIA, gravity=GRAV[11], mu=MU, fz_max=FZ_MAX, w_state=Q_W,
          w_force=R_W):
    """Forces (12, NH) of the reference's MPC for one problem.  The keyword constants default to the reference's (module
    constants above); they are the call arguments of optistate_b200.mpc.mpc_forces of the same names."""
    H, g, _ = build_qp(x, body_ref, p, dt, mass=mass, inertia=inertia, gravity=gravity, w_state=w_state, w_force=w_force)
    A, b, pinned = constraints(contact, mu=mu, fz_max=fz_max)
    return solve_ldp(H, g, A, b, pinned).reshape(NH, 12).T
