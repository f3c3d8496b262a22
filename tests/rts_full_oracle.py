"""TEST INFRASTRUCTURE ONLY - NumPy restatement of the full-covariance smoother (DESIGN.md section 0.2), on top of
tests/rts_oracle.py: the same recursion and certificate with the transition of either covariance model.

transition():       F_d of step t's predict: I + dt F with R(x+_{t-1}) (predict), or exp(dt F) element-wise with R of the step's
                    reference body angles (predict_mpc).
forward():          kf_numpy.run's filter for either model, keeping P+_t and the F_d of every step.
rts():              the backward recursion over a given F sequence, with np.linalg.solve or a Cholesky solve.
map_certificate():  the dense normal equations of rts_oracle.map_certificate over a given F sequence.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg

from oracle import kf_numpy as kn
from tests import rts_oracle as ro


def transition(x_post_prev, body_ref=None, model="predict", dt=kn.DT):
    """F_d of one predict: model "predict" from the previous posterior's attitude, "mpc" from the step's body_ref [12]."""
    if model == "predict":
        return ro.transition(x_post_prev, dt)
    F = np.zeros((12, 12))
    F[3:6, 9:12] = np.eye(3)
    F[0:3, 6:9] = kn.rot_zyx(*body_ref[0:3]).T
    return np.exp(dt * F)


def forward(stream, x0=None, P0=None, Q=None, R=None, model="predict"):
    """kf_numpy.run's recursion; returns x+ [T,12], x- [T,12], z [T,10], P+ [T,12,12] and F [T,12,12] (F[t]: step t's predict)."""
    Q = np.diag(kn.Q_DEFAULT) if Q is None else np.asarray(Q, float)
    Rn = np.diag(kn.R_DEFAULT) if R is None else np.asarray(R, float)
    x = kn.START.copy() if x0 is None else np.asarray(x0, float).reshape(12).copy()
    P = Q.copy() if P0 is None else np.asarray(P0, float).copy()
    T = stream["imu"].shape[0]
    xs, xm, zs, Ps, Fs = np.empty((T, 12)), np.empty((T, 12)), np.empty((T, 10)), np.empty((T, 12, 12)), np.empty((T, 12, 12))
    for t in range(T):
        z = kn.form_measurement(stream["imu"][t], stream["p"][t], stream["dp"][t], stream["contact"][t])
        F = transition(x, stream["body_ref"][t] if model == "mpc" else None, model)
        x_pred, _, _ = kn.propagate_mean(x, stream["p"][t], stream["f"][t])
        P = F @ P @ F.T + Q
        x, P, *_ = kn.joint_update(x_pred, P, z, Rn)
        xs[t], xm[t], zs[t], Ps[t], Fs[t] = x, x_pred, z, P, F
    return dict(x=xs, x_model=xm, z=zs, P=Ps, F=Fs)


def transitions(x_post, model="predict", body_ref=None, x0=None):
    """F [T,12,12] of the steps of a filter run from its posteriors (predict) or reference angles [T,12] (mpc)."""
    T = x_post.shape[0]
    x_prev = np.concatenate([np.asarray(kn.START if x0 is None else x0, float).reshape(1, 12), x_post[:-1]])
    return np.stack([transition(x_prev[t], None if body_ref is None else body_ref[t], model) for t in range(T)]) if T else np.empty((0, 12, 12))


def rts(x_post, x_prior, P_post, Q, F, solver="solve"):
    """Backward recursion with P-_{t+1} = F[t+1] P+_t F[t+1]^T + Q; returns (xs [T,12], Ps [T,12,12])."""
    T = x_post.shape[0]
    xs, Ps = np.empty_like(x_post), np.empty_like(P_post)
    if T == 0:
        return xs, Ps
    xs[-1], Ps[-1] = x_post[-1], P_post[-1]
    for t in range(T - 2, -1, -1):
        Ft = F[t + 1]
        Pm = Ft @ P_post[t] @ Ft.T + Q
        C = Ft @ P_post[t]
        G = (np.linalg.solve(Pm, C) if solver == "solve" else scipy.linalg.cho_solve(scipy.linalg.cho_factor(Pm, lower=True), C)).T
        xs[t] = x_post[t] + G @ (xs[t + 1] - x_prior[t + 1])
        Ps[t] = P_post[t] + G @ (Ps[t + 1] - Pm) @ G.T
    return xs, Ps


def map_certificate(x0, P0, Q, R, x_post, x_prior, z, F):
    """rts_oracle.map_certificate with F[t] as step t's transition (F[0] acts on x0)."""
    T, n = x_post.shape[0], 12
    H = np.zeros((10, 12))
    H[np.arange(10), kn.SEL] = 1.0
    Qi, Ri = np.linalg.inv(Q), np.linalg.inv(R)
    A = np.zeros((n * T, n * T))
    b = np.zeros(n * T)
    blk = lambda t: slice(n * t, n * t + n)  # noqa: E731
    Pm0i = np.linalg.inv(F[0] @ P0 @ F[0].T + Q)
    A[blk(0), blk(0)] += Pm0i
    b[blk(0)] += Pm0i @ x_prior[0]
    for t in range(T - 1):
        Ft = F[t + 1]
        c = x_prior[t + 1] - Ft @ x_post[t]
        A[blk(t + 1), blk(t + 1)] += Qi
        A[blk(t + 1), blk(t)] -= Qi @ Ft
        A[blk(t), blk(t + 1)] -= Ft.T @ Qi
        A[blk(t), blk(t)] += Ft.T @ Qi @ Ft
        b[blk(t + 1)] += Qi @ c
        b[blk(t)] -= Ft.T @ Qi @ c
    for t in range(T):
        A[blk(t), blk(t)] += H.T @ Ri @ H
        b[blk(t)] += H.T @ Ri @ z[t]
    Ainv = np.linalg.inv(A)
    return (Ainv @ b).reshape(T, n), np.stack([Ainv[blk(t), blk(t)] for t in range(T)])


def rel_errors(xs, Ps_or_var, xs_ref, var_ref):
    """Largest error of x and of var relative to each state's largest |value| over the steps."""
    var = np.einsum("tii->ti", Ps_or_var) if Ps_or_var.ndim == 3 else Ps_or_var
    sx = np.abs(xs_ref).max(axis=0)
    sv = np.abs(var_ref).max(axis=0)
    ex = float((np.abs(xs - xs_ref).max(axis=0) / np.where(sx > 0, sx, 1.0)).max())
    ev = float((np.abs(var - var_ref).max(axis=0) / np.where(sv > 0, sv, 1.0)).max())
    return ex, ev
