"""TEST INFRASTRUCTURE ONLY - NumPy restatement of the E-step of EM for diagonal Q and R (DESIGN.md section 0), independent of the
closed forms the CUDA kernel uses.

The model extends the smoother's one step back: x_{-1} ~ N(x0, P0), x_{t+1} = x-_{t+1} + F_{t+1} (x_t - x+_t) + w_t for
t = -1 .. T-2 (x+_{-1} = x0), z_t = H x_t + v_t.  Arrays of the extended chain are indexed k = t + 1: Xp[k] = x+_{k-1}
(Xp[0] = x0), PP[k] = P+_{k-1} (PP[0] = P0), and Fs[k] / xm[k] are the transition and prior mean into step k.

forward():          rts_oracle.forward's filter with optional caller-supplied z, returning the extended chain.
linear_forward():   the same filter on a frozen affine model (given Fs and offsets), for the EM monotonicity check.
estep_textbook():   RTS with the lag-one covariance P_{k+1,k|T} = Ps_{k+1} G_k^T, then E[w w^T] and E[v v^T] from their definitions;
                    the log-likelihood from the filter's innovations.
estep_dense():      the same three sums from the dense joint posterior over all 12 (T+1) unknowns and the dense marginal of the
                    stacked 10 T measurements.
em():               the EM loop (per trajectory or pooled), re-running the forward pass every iteration.
"""
from __future__ import annotations

import numpy as np

from oracle import kf_numpy as kn
from tests import rts_oracle as ro

H = np.zeros((10, 12))
H[np.arange(10), kn.SEL] = 1.0
LOG_2PI = np.log(2.0 * np.pi)


def forward(stream, x0=None, P0=None, Q=None, R=None, z=None):
    """Extended chain of the filter (predict() model): dict(Xp [T+1,12], PP [T+1,12,12], xm [T,12], Fs [T,12,12], z [T,10])."""
    Q = np.diag(kn.Q_DEFAULT) if Q is None else np.asarray(Q, float)
    Rn = np.diag(kn.R_DEFAULT) if R is None else np.asarray(R, float)
    x = kn.START.copy() if x0 is None else np.asarray(x0, float).reshape(12).copy()
    P = Q.copy() if P0 is None else np.asarray(P0, float).copy()
    T = stream["p"].shape[0]
    Xp, PP, xm, zs = [x.copy()], [P.copy()], np.empty((T, 12)), np.empty((T, 10))
    for t in range(T):
        zt = kn.form_measurement(stream["imu"][t], stream["p"][t], stream["dp"][t], stream["contact"][t]) if z is None else z[t]
        x_pred, _, Rm = kn.propagate_mean(x, stream["p"][t], stream["f"][t])
        P = kn.propagate_cov(P, Rm, Q)
        x, P, *_ = kn.joint_update(x_pred, P, zt, Rn)
        xm[t], zs[t] = x_pred, zt
        Xp.append(x)
        PP.append(P)
    Xp, PP = np.array(Xp), np.array(PP)
    Fs = np.array([ro.transition(Xp[k]) for k in range(T)]).reshape(T, 12, 12)
    return dict(Xp=Xp, PP=PP, xm=xm, Fs=Fs, z=zs)


def linear_forward(Fs, c, x0, P0, Q, R, z):
    """Kalman filter of the affine model x_k = Fs[k-1] x_{k-1} + c[k-1] + w (extended indices), z = H x + v."""
    T = z.shape[0]
    x, P = np.asarray(x0, float).copy(), np.asarray(P0, float).copy()
    Xp, PP, xm = [x.copy()], [P.copy()], np.empty((T, 12))
    for k in range(T):
        x = Fs[k] @ x + c[k]
        P = Fs[k] @ P @ Fs[k].T + Q
        xm[k] = x
        S = H @ P @ H.T + R
        K = np.linalg.solve(S, H @ P).T
        x = x + K @ (z[k] - H @ x)
        P = P - K @ S @ K.T
        P = 0.5 * (P + P.T)
        Xp.append(x.copy())
        PP.append(P.copy())
    return dict(Xp=np.array(Xp), PP=np.array(PP), xm=xm, Fs=np.asarray(Fs), z=z)


def estep_textbook(ch, Q, R):
    """(Sw [12], Sv [10], loglik) of one trajectory."""
    Xp, PP, xm, Fs, z = ch["Xp"], ch["PP"], ch["xm"], ch["Fs"], ch["z"]
    T = z.shape[0]
    xs, Ps = np.empty_like(Xp), np.empty_like(PP)
    Pc = np.empty((T, 12, 12))  # Cov(x_{k+1}, x_k | Z)
    xs[T], Ps[T] = Xp[T], PP[T]
    ll = 0.0
    for k in range(T - 1, -1, -1):
        F = Fs[k]
        Pm = F @ PP[k] @ F.T + Q
        G = np.linalg.solve(Pm, F @ PP[k]).T
        xs[k] = Xp[k] + G @ (xs[k + 1] - xm[k])
        Ps[k] = PP[k] + G @ (Ps[k + 1] - Pm) @ G.T
        Pc[k] = Ps[k + 1] @ G.T
        S = H @ Pm @ H.T + R
        y = z[k] - H @ xm[k]
        ll += -0.5 * (10 * LOG_2PI + np.linalg.slogdet(S)[1] + y @ np.linalg.solve(S, y))
    Sw, Sv = np.zeros(12), np.zeros(10)
    for k in range(T):
        F = Fs[k]
        mw = xs[k + 1] - xm[k] - F @ (xs[k] - Xp[k])
        Cw = Ps[k + 1] - F @ Pc[k].T - Pc[k] @ F.T + F @ Ps[k] @ F.T
        Sw += mw ** 2 + np.diag(Cw)
        Sv += (z[k] - H @ xs[k + 1]) ** 2 + np.diag(H @ Ps[k + 1] @ H.T)
    return Sw, Sv, ll


def estep_dense(ch, Q, R):
    """The same sums from the dense posterior over x_{-1} .. x_{T-1} and the dense likelihood of the stacked measurements."""
    Xp, PP, xm, Fs, z = ch["Xp"], ch["PP"], ch["xm"], ch["Fs"], ch["z"]
    T, n = z.shape[0], 12
    U = T + 1
    blk = lambda k: slice(n * k, n * k + n)  # noqa: E731
    A0, b0 = np.zeros((n * U, n * U)), np.zeros(n * U)  # prior precision of the chain, without the measurements
    P0i = np.linalg.inv(PP[0])
    A0[blk(0), blk(0)] += P0i
    b0[blk(0)] += P0i @ Xp[0]
    Qi, Ri = np.linalg.inv(Q), np.linalg.inv(R)
    cs = [xm[k] - Fs[k] @ Xp[k] for k in range(T)]
    for k in range(T):
        F, c = Fs[k], cs[k]
        A0[blk(k + 1), blk(k + 1)] += Qi
        A0[blk(k + 1), blk(k)] -= Qi @ F
        A0[blk(k), blk(k + 1)] -= F.T @ Qi
        A0[blk(k), blk(k)] += F.T @ Qi @ F
        b0[blk(k + 1)] += Qi @ c
        b0[blk(k)] -= F.T @ Qi @ c
    A, b = A0.copy(), b0.copy()
    for k in range(1, U):
        A[blk(k), blk(k)] += H.T @ Ri @ H
        b[blk(k)] += H.T @ Ri @ z[k - 1]
    C = np.linalg.inv(A)
    m = (C @ b).reshape(U, n)
    Sw, Sv = np.zeros(12), np.zeros(10)
    for k in range(T):
        F = Fs[k]
        mw = m[k + 1] - F @ m[k] - cs[k]
        J = np.hstack([-F, np.eye(12)])
        Sw += mw ** 2 + np.diag(J @ C[n * k:n * k + 2 * n, n * k:n * k + 2 * n] @ J.T)
        Sv += (z[k] - H @ m[k + 1]) ** 2 + np.diag(H @ C[blk(k + 1), blk(k + 1)] @ H.T)
    Sig = np.linalg.inv(A0)
    mu = Sig @ b0
    Hb = np.zeros((10 * T, n * U))
    for k in range(1, U):
        Hb[10 * (k - 1):10 * k, blk(k)] = H
    Sz = Hb @ Sig @ Hb.T + np.kron(np.eye(T), R)
    yz = z.reshape(-1) - Hb @ mu
    ll = -0.5 * (10 * T * LOG_2PI + np.linalg.slogdet(Sz)[1] + yz @ np.linalg.solve(Sz, yz))
    return Sw, Sv, ll


def em(streams, q, r, iters, shared, x0=None, P0=None, zs=None):
    """EM over a list of streams ([T, C] arrays each; zs: optional caller-supplied z per stream).  q [n_traj, 12], r [n_traj, 10]
    per trajectory (or [12] / [10] with shared).  P0 None is held at the starting Q.  Returns (q, r, loglik [iters, n_traj])."""
    n = len(streams)
    T = streams[0]["p"].shape[0]
    q = np.array(q, float)
    r = np.array(r, float)
    qs = np.broadcast_to(q, (n, 12)).copy()
    P0s = [np.diag(qs[j]) if P0 is None else np.asarray(P0, float) for j in range(n)]
    lls = []
    for _ in range(iters):
        qj = np.broadcast_to(q, (n, 12)) if shared else q
        rj = np.broadcast_to(r, (n, 10)) if shared else r
        stats = []
        for j in range(n):
            Q, Rn = np.diag(qj[j]), np.diag(rj[j])
            ch = forward(streams[j], x0, P0s[j], Q, Rn, None if zs is None else zs[j])
            stats.append(estep_textbook(ch, Q, Rn))
        lls.append([s[2] for s in stats])
        Sw = np.array([s[0] for s in stats])
        Sv = np.array([s[1] for s in stats])
        if shared:
            q, r = Sw.sum(0) / (n * T), Sv.sum(0) / (n * T)
        else:
            q, r = Sw / T, Sv / T
    return q, r, np.array(lls)


def simulate(seed, T, q_true, r_true):
    """A stream of synth.make_stream whose state follows the mean model plus N(0, q_true) noise, and z = H x + N(0, r_true)."""
    from optistate_b200.synth import make_stream

    st = make_stream(seed, T)
    rng = np.random.default_rng(seed + 99)
    x = kn.START.copy()
    zs = np.empty((T, 10))
    for t in range(T):
        x = kn.propagate_mean(x, st["p"][t], st["f"][t])[0] + np.sqrt(q_true) * rng.standard_normal(12)
        zs[t] = H @ x + np.sqrt(r_true) * rng.standard_normal(10)
    return st, zs
