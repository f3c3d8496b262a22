"""TEST INFRASTRUCTURE ONLY - NumPy restatement of the fixed-interval Rauch-Tung-Striebel smoother (DESIGN.md section 0).

forward():          the filter of oracle/kf_numpy.run, step for step with the same functions, that also keeps P+_t of every step.
rts():              the textbook backward recursion on full 12x12 matrices with np.linalg.solve.
map_certificate():  a solver-independent check for short recordings: the MAP estimate of the affine model
                        x_0 ~ N(x-_0, P-_0),  x_{t+1} = x-_{t+1} + F_{t+1} (x_t - x+_t) + w_t,  w_t ~ N(0, Q),  z_t = H x_t + v_t,  v_t ~ N(0, R)
                    from its dense normal equations over all 12 T unknowns.  The smoother of the filter that ran is exactly this MAP
                    estimate; its covariances are the diagonal blocks of the inverse normal matrix.
"""
from __future__ import annotations

import numpy as np

from oracle import kf_numpy as kn


def transition(x_post_prev, dt=kn.DT):
    """F_d = I + dt F of the predict() covariance model, F[0:3,6:9] = R(x+)^T, F[3:6,9:12] = I (un-truncated)."""
    F = np.eye(12)
    F[0:3, 6:9] += dt * kn.rot_zyx(*x_post_prev[0:3]).T
    F[3:6, 9:12] += dt * np.eye(3)
    return F


def forward(stream, x0=None, P0=None, Q=None, R=None):
    """kf_numpy.run's recursion (predict() model) returning x+ [T,12], x- [T,12], z [T,10], P+ [T,12,12]."""
    Q = np.diag(kn.Q_DEFAULT) if Q is None else np.asarray(Q, float)
    Rn = np.diag(kn.R_DEFAULT) if R is None else np.asarray(R, float)
    x = kn.START.copy() if x0 is None else np.asarray(x0, float).reshape(12).copy()
    P = Q.copy() if P0 is None else np.asarray(P0, float).copy()
    T = stream["imu"].shape[0]
    xs, xm, zs, Ps = np.empty((T, 12)), np.empty((T, 12)), np.empty((T, 10)), np.empty((T, 12, 12))
    for t in range(T):
        z = kn.form_measurement(stream["imu"][t], stream["p"][t], stream["dp"][t], stream["contact"][t])
        x_pred, _, Rm = kn.propagate_mean(x, stream["p"][t], stream["f"][t])
        P = kn.propagate_cov(P, Rm, Q)
        x, P, *_ = kn.joint_update(x_pred, P, z, Rn)
        xs[t], xm[t], zs[t], Ps[t] = x, x_pred, z, P
    return dict(x=xs, x_model=xm, z=zs, P=Ps)


def rts(x_post, x_prior, P_post, Q, dt=kn.DT):
    """Backward recursion; returns (xs [T,12], Ps [T,12,12])."""
    T = x_post.shape[0]
    xs, Ps = np.empty_like(x_post), np.empty_like(P_post)
    if T == 0:
        return xs, Ps
    xs[-1], Ps[-1] = x_post[-1], P_post[-1]
    for t in range(T - 2, -1, -1):
        F = transition(x_post[t], dt)
        Pm = F @ P_post[t] @ F.T + Q
        G = np.linalg.solve(Pm, F @ P_post[t]).T  # G = P+ F^T Pm^-1 (Pm symmetric)
        xs[t] = x_post[t] + G @ (xs[t + 1] - x_prior[t + 1])
        Ps[t] = P_post[t] + G @ (Ps[t + 1] - Pm) @ G.T
    return xs, Ps


def map_certificate(x0, P0, Q, R, x_post, x_prior, z, dt=kn.DT):
    """Mean [T,12] and marginal covariances [T,12,12] of the affine model above, from its dense normal equations."""
    T, n = x_post.shape[0], 12
    H = np.zeros((10, 12))
    H[np.arange(10), kn.SEL] = 1.0
    Qi, Ri = np.linalg.inv(Q), np.linalg.inv(R)
    F0 = transition(np.asarray(x0, float).reshape(12), dt)
    Pm0 = F0 @ P0 @ F0.T + Q
    A = np.zeros((n * T, n * T))
    b = np.zeros(n * T)
    blk = lambda t: slice(n * t, n * t + n)  # noqa: E731
    # prior on x_0
    P0i = np.linalg.inv(Pm0)
    A[blk(0), blk(0)] += P0i
    b[blk(0)] += P0i @ x_prior[0]
    # process terms  r = x_{t+1} - F x_t - c,  c = x-_{t+1} - F x+_t
    for t in range(T - 1):
        F = transition(x_post[t], dt)
        c = x_prior[t + 1] - F @ x_post[t]
        A[blk(t + 1), blk(t + 1)] += Qi
        A[blk(t + 1), blk(t)] -= Qi @ F
        A[blk(t), blk(t + 1)] -= F.T @ Qi
        A[blk(t), blk(t)] += F.T @ Qi @ F
        b[blk(t + 1)] += Qi @ c
        b[blk(t)] -= F.T @ Qi @ c
    # measurements
    for t in range(T):
        A[blk(t), blk(t)] += H.T @ Ri @ H
        b[blk(t)] += H.T @ Ri @ z[t]
    Ainv = np.linalg.inv(A)
    mean = (Ainv @ b).reshape(T, n)
    cov = np.stack([Ainv[blk(t), blk(t)] for t in range(T)])
    return mean, cov
