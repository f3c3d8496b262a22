"""TEST INFRASTRUCTURE ONLY - NumPy restatement of the adjoint of the decoupled-group filter (DESIGN.md section 0.4).

moments():  the leg moments C [T, 9] (C[3m + k] = sum_l p_l[m] f_l[k]) of the mean model, as the measurement pre-pass forms them.
mean_jac(): J = dx-/dx+ of the mean model the filter kernels evaluate, w' = w + R diag(dt / I) g(R), g_i = eps_ijk (C R)_jk,
            th' = th + dt trunc(R^T) w; trunc(R^T) is piecewise constant and contributes no derivative.
adjoint():  the reverse recursion of include/optistate_kf.h, one decoupled group at a time, fed a forward chain (x+, x-, P+ of
            every step, z and C) the way rts_oracle and em_oracle are fed; returns grad [46] (q_bar, r_bar, x0_bar, diag P0_bar).
"""
from __future__ import annotations

import numpy as np

from oracle import kf_numpy as kn
from tests import rts_oracle as ro

GROUPS = ([0, 1, 2, 6, 7, 8], [3, 9], [4, 10], [5, 11])
SEL = list(kn.SEL)


def moments(p, f):
    """p, f [T, 12] -> C [T, 9]."""
    P, Fv = p.reshape(-1, 4, 3), f.reshape(-1, 4, 3)
    return np.einsum("tlm,tlk->tmk", P, Fv).reshape(-1, 9)


def rot_derivs(th):
    """dR/dth_m [3, 3, 3] (m first) of R = Rz(c) Ry(b) Rx(a)."""
    a, b, c = th
    R = kn.rot_zyx(a, b, c)
    X = np.array([[0, 0, 0], [0, 0, -1], [0, 1, 0]], float)
    Z = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 0]], float)
    Rz = np.array([[np.cos(c), -np.sin(c), 0], [np.sin(c), np.cos(c), 0], [0, 0, 1]])
    Rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    dRy = np.array([[-np.sin(b), 0, np.cos(b)], [0, 0, 0], [-np.cos(b), 0, -np.sin(b)]])
    return R, np.stack([R @ X, Rz @ dRy @ Rx, Z @ R])


def _g(C, M):
    CM = C.reshape(3, 3) @ M
    return np.array([CM[1, 2] - CM[2, 1], CM[2, 0] - CM[0, 2], CM[0, 1] - CM[1, 0]])


def mean_jac(x_post_prev, C, dt=kn.DT, inertia=kn.INERTIA):
    R, dR = rot_derivs(x_post_prev[0:3])
    d = dt / inertia
    u = d * _g(C, R)
    J = np.eye(12)
    J[3:6, 9:12] += dt * np.eye(3)
    for m in range(3):
        J[6:9, m] = dR[m] @ u + R @ (d * _g(C, dR[m]))
    Tm = np.trunc(R.T)
    if np.any(Tm != 0):
        J[0:3, 6:9] += dt * Tm
    return J, dR


def adjoint(x_post, x_prior, P_post, z, C, x_bar, x0, P0, q, r, dt=kn.DT, inertia=kn.INERTIA):
    """x_post, x_prior, x_bar [T, 12]; P_post [T, 12, 12]; z [T, 10]; C [T, 9]; x0 [12]; P0 [12, 12]; q [12], r [10]."""
    T = x_post.shape[0]
    qb, rb = np.zeros(12), np.zeros(10)
    a = np.zeros(12)
    Pi = np.zeros((12, 12))
    Q = np.diag(q)
    for t in range(T - 1, -1, -1):
        xp = x0 if t == 0 else x_post[t - 1]
        Pp = P0 if t == 0 else P_post[t - 1]
        a = a + x_bar[t]
        F = ro.transition(xp, dt)
        Pm = F @ Pp @ F.T + Q
        J, dR = mean_jac(xp, C[t], dt, inertia)
        a_new = np.zeros(12)
        Pi_new = np.zeros((12, 12))
        for I in GROUPS:
            Ig = [s for s in I if s in SEL]
            rows = [SEL.index(s) for s in Ig]
            n, m = len(I), len(Ig)
            H = np.zeros((m, n))
            for j, s in enumerate(Ig):
                H[j, I.index(s)] = 1.0
            Pg, Fg, Pig, ag = Pm[np.ix_(I, I)], F[np.ix_(I, I)], Pi[np.ix_(I, I)], a[I]
            S = H @ Pg @ H.T + np.diag(r[rows])
            Si = np.linalg.inv(S)
            K = Pg @ H.T @ Si
            A = np.eye(n) - K @ H
            v = Si @ (z[t, rows] - x_prior[t, Ig])
            b = K.T @ ag
            rb[rows] += np.diag(K.T @ Pig @ K) - b * v
            M = A.T @ np.outer(ag, H.T @ v)
            Pb = A.T @ Pig @ A + 0.5 * (M + M.T)
            qb[I] += np.diag(Pb)
            Pi_new[np.ix_(I, I)] = Fg.T @ Pb @ Fg
            at = A.T @ ag
            a_new[I] = J[np.ix_(I, I)].T @ at
            if I[0] == 0:  # the th-term of F: dF[j][w] = dt dR[w][j]
                B = 2.0 * (Pb @ Fg @ Pp[np.ix_(I, I)])[0:3, 3:6]
                for mm in range(3):
                    a_new[mm] += dt * np.sum(B * dR[mm].T)
        a, Pi = a_new, Pi_new
    return np.concatenate([qb, rb, a, np.diag(Pi)])
