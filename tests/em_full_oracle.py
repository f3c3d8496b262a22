"""TEST INFRASTRUCTURE ONLY - the extended chain of the EM E-step (tests/em_oracle.py, DESIGN.md section 0.1) for either covariance
model of the full-covariance smoother (tests/rts_full_oracle.py, DESIGN.md section 0.3).

The model x_{-1} ~ N(x0, P0), x_{t+1} = x-_{t+1} + F_{t+1} (x_t - x+_t) + w_t, z_t = H x_t + v_t does not depend on which F is used,
so em_oracle.estep_textbook and em_oracle.estep_dense take this module's chains unchanged (estep_dense's log-likelihood excepted
under predict_mpc: see loglik_dense).

forward():          the filter of either model (rts_full_oracle.transition), optional caller-supplied z, as an extended chain:
                    Xp [T+1,12], PP [T+1,12,12], xm [T,12], Fs [T,12,12] (Fs[0] from x0, or from body_ref[0] under mpc), z [T,10].
loglik_dense():     the log-likelihood from the dense joint posterior alone (the certificate for predict_mpc, whose chain prior
                    em_oracle.estep_dense cannot invert).
estep_cholesky():   em_oracle.estep_textbook with Cholesky solves in place of LU, to compare two solvers where the certificate is
                    ill-conditioned.
em():               the NumPy EM loop over either model (em_oracle.em knows the predict() model only).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg

from oracle import kf_numpy as kn
from tests import em_oracle as eo
from tests import rts_full_oracle as rf


def forward(stream, x0=None, P0=None, Q=None, R=None, model="predict", z=None):
    """Extended chain of the filter of `model` ("predict" or "mpc"; mpc reads stream["body_ref"] [T,12])."""
    Q = np.diag(kn.Q_DEFAULT) if Q is None else np.asarray(Q, float)
    Rn = np.diag(kn.R_DEFAULT) if R is None else np.asarray(R, float)
    x = kn.START.copy() if x0 is None else np.asarray(x0, float).reshape(12).copy()
    P = Q.copy() if P0 is None else np.asarray(P0, float).copy()
    T = stream["p"].shape[0]
    Xp, PP, xm, zs, Fs = [x.copy()], [P.copy()], np.empty((T, 12)), np.empty((T, 10)), np.empty((T, 12, 12))
    for t in range(T):
        zt = kn.form_measurement(stream["imu"][t], stream["p"][t], stream["dp"][t], stream["contact"][t]) if z is None else z[t]
        F = rf.transition(x, stream["body_ref"][t] if model == "mpc" else None, model)
        x_pred, _, _ = kn.propagate_mean(x, stream["p"][t], stream["f"][t])
        P = F @ P @ F.T + Q
        x, P, *_ = kn.joint_update(x_pred, P, zt, Rn)
        xm[t], zs[t], Fs[t] = x_pred, zt, F
        Xp.append(x)
        PP.append(P)
    return dict(Xp=np.array(Xp), PP=np.array(PP), xm=xm, Fs=Fs, z=zs)


def estep_cholesky(ch, Q, R):
    """(Sw [12], Sv [10], loglik) as estep_textbook computes them, with G and the innovation solved by Cholesky."""
    Xp, PP, xm, Fs, z = ch["Xp"], ch["PP"], ch["xm"], ch["Fs"], ch["z"]
    H = eo.H
    T = z.shape[0]
    xs, Ps, Pc = np.empty_like(Xp), np.empty_like(PP), np.empty((T, 12, 12))
    xs[T], Ps[T] = Xp[T], PP[T]
    ll = 0.0
    for k in range(T - 1, -1, -1):
        F = Fs[k]
        Pm = F @ PP[k] @ F.T + Q
        G = scipy.linalg.cho_solve(scipy.linalg.cho_factor(Pm, lower=True), F @ PP[k]).T
        xs[k] = Xp[k] + G @ (xs[k + 1] - xm[k])
        Ps[k] = PP[k] + G @ (Ps[k + 1] - Pm) @ G.T
        Pc[k] = Ps[k + 1] @ G.T
        c, low = scipy.linalg.cho_factor(H @ Pm @ H.T + R, lower=True)
        y = z[k] - H @ xm[k]
        ll += -0.5 * (10 * eo.LOG_2PI + 2.0 * np.log(np.diag(c)).sum() + y @ scipy.linalg.cho_solve((c, low), y))
    Sw, Sv = np.zeros(12), np.zeros(10)
    for k in range(T):
        F = Fs[k]
        mw = xs[k + 1] - xm[k] - F @ (xs[k] - Xp[k])
        Cw = Ps[k + 1] - F @ Pc[k].T - Pc[k] @ F.T + F @ Ps[k] @ F.T
        Sw += mw ** 2 + np.diag(Cw)
        Sv += (z[k] - H @ xs[k + 1]) ** 2 + np.diag(H @ Ps[k + 1] @ H.T)
    return Sw, Sv, ll


def loglik_dense(ch, Q, R):
    """log p(z) from the dense joint posterior alone: log p(m) + log p(z | m) - log p(m | z) at its mean m, with the chain's prior
    density written out transition by transition.  em_oracle.estep_dense inverts the chain's prior precision instead, which under
    predict_mpc (F_d = 1 1^T + D, largest eigenvalue ~12) grows like 12^(2T) and is meaningless at T = 40."""
    Xp, PP, xm, Fs, z = ch["Xp"], ch["PP"], ch["xm"], ch["Fs"], ch["z"]
    H, T, n = eo.H, z.shape[0], 12
    U = T + 1
    blk = lambda k: slice(n * k, n * k + n)  # noqa: E731
    Qi, Ri, P0i = np.linalg.inv(Q), np.linalg.inv(R), np.linalg.inv(PP[0])
    cs = [xm[k] - Fs[k] @ Xp[k] for k in range(T)]
    A, b = np.zeros((n * U, n * U)), np.zeros(n * U)
    A[blk(0), blk(0)] += P0i
    b[blk(0)] += P0i @ Xp[0]
    for k in range(T):
        F, c = Fs[k], cs[k]
        A[blk(k + 1), blk(k + 1)] += Qi + H.T @ Ri @ H
        A[blk(k + 1), blk(k)] -= Qi @ F
        A[blk(k), blk(k + 1)] -= F.T @ Qi
        A[blk(k), blk(k)] += F.T @ Qi @ F
        b[blk(k + 1)] += Qi @ c + H.T @ Ri @ z[k]
        b[blk(k)] -= F.T @ Qi @ c
    m = np.linalg.solve(A, b).reshape(U, n)

    def log_normal(e, C):
        return -0.5 * (len(e) * eo.LOG_2PI + np.linalg.slogdet(C)[1] + e @ np.linalg.solve(C, e))

    lp = log_normal(m[0] - Xp[0], PP[0]) + sum(log_normal(m[k + 1] - Fs[k] @ m[k] - cs[k], Q) for k in range(T))
    lz = sum(log_normal(z[k] - H @ m[k + 1], R) for k in range(T))
    return lp + lz + 0.5 * (n * U * eo.LOG_2PI - np.linalg.slogdet(A)[1])


def em(streams, q, r, iters, shared, x0=None, P0=None, zs=None, model="predict"):
    """em_oracle.em over the filter of `model` (streams carry body_ref under mpc).  Returns (q, r, loglik [iters, n_traj])."""
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
            ch = forward(streams[j], x0, P0s[j], Q, Rn, model, None if zs is None else zs[j])
            stats.append(eo.estep_textbook(ch, Q, Rn))
        lls.append([s[2] for s in stats])
        Sw = np.array([s[0] for s in stats])
        Sv = np.array([s[1] for s in stats])
        if shared:
            q, r = Sw.sum(0) / (n * T), Sv.sum(0) / (n * T)
        else:
            q, r = Sw / T, Sv / T
    return q, r, np.array(lls)
