"""Batched convex force MPC - SURVEY 8(f) row 3: the QP `Kalman_Filter.predict_mpc` solves for its ground-reaction
forces (/root/reference/misc/force_controller.py:15-225, set up by /root/reference/kalman_filter/kalman_filter.py:64-77,
140-152), one problem per warp on the device (csrc/kf_mpc.cuh).  The reference uses CasADi + qpOASES; neither exists
offline and no reference test pins a force vector, so parity is anchored on the uniqueness of the minimiser of this
strictly convex QP (tests: KKT optimality + an independent active-set solve).  FP64 only.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as nv
from .settings import INITIAL_PARAMS

HORIZON = 5
# kalman_filter.py:64-70 (Q = P) and force_controller.py:149-151
W_STATE = (10.0, 10.0, 10.0, 100.0, 100.0, 100.0, 1.0, 1.0, 5.0, 1.0, 1.0, 1.0)
W_FORCE = 1e-6
MU = 0.6
FZ_MAX = 150.0
ST_IPM_LIMIT, ST_UNPOLISHED, ST_TOO_MANY_LEGS, ST_WARM = 1, 2, 4, 8


def _dev64(a, device):
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
    return t.to(device=device, dtype=torch.float64).contiguous()


def mpc_forces(x, body_ref, p, contact, *, dt: float = INITIAL_PARAMS.DT_mpc, mass: float = INITIAL_PARAMS.ROBOT_MASS, inertia=None,
               gravity: float = INITIAL_PARAMS.GRAVITY, mu: float = MU, fz_max: float = FZ_MAX, w_state=W_STATE, w_force: float = W_FORCE,
               max_free_legs=None, device=None, warm=None, solver: str = "auto", max_changes: int = 0):
    """Solves N force MPC problems.

    x [12, N] current states; body_ref [5, 12, N] reference states of the horizon; p [12, N] body-frame feet;
    contact [4, N] (0 swing, 1 stance).  max_free_legs: bound on the legs out of swing in any problem (None = taken from
    `contact`, which costs one small reduction and a host sync; it sizes the kernel's shared memory).
    solver: "auto" - the dual active-set kernels (csrc/kf_mpc_gi.cuh: one warp per problem for at most two legs out of swing, two
    warps for three and four), with the interior-point kernel (csrc/kf_mpc.cuh) behind them for problems they give up on;
    "interior_point" - the interior-point kernel only, for every leg count (it takes no warm start).
    max_changes: cap on the constraints the dual active-set method may enter + drop per problem before it hands the problem to the
    interior point (0 = the kernel's default, 400).
    warm: a `WarmStart` (in / out) carrying the active set and multipliers from one solve to the next one of the same
    problems (closed loops); a set that no longer verifies falls back to the cold path inside the kernel.
    Returns (forces [5, 12, N] - stage 0 is what predict_mpc applies -, status [N]: ST_* bits | interior-point iterations << 8).
    """
    nv.require_cuda()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    x_t, p_t, c_t, b_t = _dev64(x, device), _dev64(p, device), _dev64(contact, device), _dev64(body_ref, device)
    n = x_t.shape[-1] if x_t.dim() == 2 else 1
    x_t, p_t, c_t, b_t = x_t.reshape(12, n), p_t.reshape(12, n), c_t.reshape(4, n), b_t.reshape(HORIZON, 12, n)
    if max_free_legs is None:
        max_free_legs = max(1, int((c_t != 0).sum(dim=0).max())) if n > 0 else 4
    forces = torch.empty((HORIZON, 12, n), dtype=torch.float64, device=device)
    status = torch.zeros(n, dtype=torch.int32, device=device)
    inertia = np.diag(INITIAL_PARAMS.INERTIA_ROT) if inertia is None else np.asarray(inertia, float).reshape(3)
    consts = dict(dt=float(dt), mass=float(mass), inertia0=float(inertia[0]), inertia1=float(inertia[1]), inertia2=float(inertia[2]),
                  gravity=float(gravity), mu=float(mu), fz_max=float(fz_max), w_force=float(w_force))
    if solver not in ("auto", "interior_point"):
        raise ValueError("solver must be 'auto' or 'interior_point'")
    consts["solver"] = 1.0 if solver == "interior_point" else 0.0
    consts["max_changes"] = float(max_changes)
    tensors = dict(x=x_t, body_ref=b_t, p=p_t, contact=c_t, forces=forces, status=status)
    if warm is not None:
        if warm.n != n or warm.active.device != device:
            raise ValueError("warm start was set up for another batch size or device")
        tensors.update(warm_set=warm.active, warm_mult=warm.multipliers)
    with torch.cuda.device(device):
        nv.check(int(nv.ext().kf_mpc_forces(n, int(max_free_legs), consts, [float(w) for w in w_state], tensors)), "optistate_kf_mpc_forces")
    return forces, status


class WarmStart:
    """Active set and multipliers carried between consecutive solves of the same N problems (include/optistate_kf.h,
    OptiKfMpcDesc.warm_set / warm_mult).  Starts empty: the first solve is a cold one."""

    def __init__(self, n: int, device=None):
        nv.require_cuda()
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n = int(n)
        self.active = torch.zeros((HORIZON, self.n), dtype=torch.int32, device=device)
        self.multipliers = torch.zeros((HORIZON * 4 * 5, self.n), dtype=torch.float64, device=device)

    def reset(self):
        self.active.zero_()


def estimate_state_mpc_batch(imu, p, dp, contact, body_ref, x0=None, P0=None, Q=None, R=None, *, dt: float = INITIAL_PARAMS.DT_mpc,
                             mass: float = INITIAL_PARAMS.ROBOT_MASS, inertia=None, gravity: float = INITIAL_PARAMS.GRAVITY,
                             return_p_world: bool = False, **mpc_kw):
    """The reference's closed loop `KF.estimate_state_mpc(imu, p, dp, body_ref, contact)` (kalman_filter.py:176-182) for N
    trajectories over T steps, everything on the device: at every step the force MPC is solved for each trajectory from
    its CURRENT state estimate, then one filter step runs with those forces and the predict_mpc covariance model.

    imu [T,6,N], p [T,12,N], dp [T,12,N], contact [T,4,N], body_ref [T,5,12,N] (horizon reference of each step; the
    filter's transition uses its first column, as the class does).  x0, P0, Q, R as in kf_batch (P0 None = Q); dense Q / R or a
    non-symmetric P0 run the filter step in its joint form, like the class.  dt, mass, inertia, gravity are the model constants
    of BOTH the MPC and the filter; `mpc_kw` (mu, fz_max, w_state, w_force, max_free_legs, solver, max_changes; warm = True / False /
    a WarmStart) goes to the MPC only.  With diagonal noise and a symmetric P0 the whole loop is ONE call of the C ABI
    (optistate_kf_closed_loop: nothing between the steps goes through Python or synchronises with the host).
    Returns (x_steps [T,12,N], forces [T,12,N] - the applied stage-0 forces -, mpc_status [T,N], filter status [N]) and, with
    return_p_world, the feet rotated into the world frame [T,12,N] (the reference's in-place mutation of p, which its driver
    writes into the GRU feature rows).
    """
    from .batch import _as_device, _noise, kf_batch

    nv.require_cuda()
    device = torch.device("cuda", torch.cuda.current_device())
    imu, p, dp, contact, body_ref = (_as_device(a, torch.float64, device) for a in (imu, p, dp, contact, body_ref))
    T, N = imu.shape[0], imu.shape[2]
    x = _as_device(INITIAL_PARAMS.STARTING_STATE.reshape(12) if x0 is None else x0, torch.float64, device)
    x = x.reshape(12, 1).repeat(1, N) if x.numel() == 12 else x.reshape(12, N).clone()
    xs = torch.empty((T, 12, N), dtype=torch.float64, device=device)
    fs = torch.empty((T, 12, N), dtype=torch.float64, device=device)
    mst = torch.empty((T, N), dtype=torch.int32, device=device)
    fst = torch.zeros(N, dtype=torch.int32, device=device)
    pws = torch.empty((T, 12, N), dtype=torch.float64, device=device) if return_p_world else None
    outputs = ("x_final", "P_final", "p_world_steps") if return_p_world else ("x_final", "P_final")
    # everything that would make a step synchronise with the host is settled once, before the loop: the classification of the
    # noise arguments (a dense matrix that is exactly diagonal becomes a diagonal), the symmetry of the initial P, the bound
    # on the legs out of swing over all steps
    q_t, q_kind = _noise(INITIAL_PARAMS.Q if Q is None else Q, 12, N, "Q", torch.float64, device)
    r_t, r_kind = _noise(INITIAL_PARAMS.R if R is None else R, 10, N, "R", torch.float64, device)
    diag_noise = q_kind in (nv.MAT_DIAG, nv.MAT_DIAG_PER) and r_kind in (nv.MAT_DIAG, nv.MAT_DIAG_PER)
    Pm, p_kind, p_sym = None, None, True
    if P0 is not None:
        Pm, p_kind = _noise(P0, 12, N, "P0", torch.float64, device)
        if p_kind in (nv.MAT_DENSE, nv.MAT_DENSE_PER):
            m = Pm.reshape(12, 12, -1)
            p_sym = bool(torch.equal(m, m.transpose(0, 1)))
    algo = "sequential" if (diag_noise and p_sym) else "joint"  # the packed-symmetric form needs diagonal noise and a symmetric P
    model = dict(dt=dt, mass=mass, inertia=inertia, gravity=gravity)
    if "max_free_legs" not in mpc_kw:
        mpc_kw["max_free_legs"] = max(1, int((contact != 0).sum(dim=1).max())) if T * N > 0 else 4
    warm = mpc_kw.pop("warm", True)  # True: carry the MPC's working set from step to step; False / None: cold solves; or a WarmStart
    if algo == "sequential" and T * N > 0 and (warm is None or isinstance(warm, bool)) \
            and set(mpc_kw) <= {"max_free_legs", "mu", "fz_max", "w_state", "w_force", "solver", "max_changes"}:
        # the whole loop in one call of the C ABI (optistate_kf_closed_loop): no Python, no host synchronisation between the steps
        ext = nv.ext()
        I3 = np.diag(INITIAL_PARAMS.INERTIA_ROT) if inertia is None else np.asarray(inertia, float).reshape(3)
        consts = dict(dt=float(dt), mass=float(mass), inertia0=float(I3[0]), inertia1=float(I3[1]), inertia2=float(I3[2]), gravity=float(gravity),
                      mu=float(mpc_kw.get("mu", MU)), fz_max=float(mpc_kw.get("fz_max", FZ_MAX)), w_force=float(mpc_kw.get("w_force", W_FORCE)))
        cfg = dict(n_traj=N, n_steps=T, max_free_legs=int(mpc_kw["max_free_legs"]), x0_per_traj=1, q_kind=q_kind, r_kind=r_kind,
                   p0_kind=nv.MAT_NONE if Pm is None else p_kind, warm_start=1 if warm is True else 0,
                   solver=1 if mpc_kw.get("solver", "auto") == "interior_point" else 0, max_changes=int(mpc_kw.get("max_changes", 0)))
        tensors = dict(imu=imu, p=p, dp=dp, contact=contact, body_ref=body_ref, x0=x.contiguous(), Q=q_t, R=r_t, x_steps=xs, forces=fs,
                       mpc_status=mst, status=fst,
                       workspace=torch.empty(int(ext.kf_closed_loop_workspace_bytes(N, T)), dtype=torch.uint8, device=device))
        if Pm is not None:
            tensors["P0"] = Pm
        if return_p_world:
            tensors["p_world_steps"] = pws
        with torch.cuda.device(device):
            nv.check(int(ext.kf_closed_loop(cfg, consts, [float(w) for w in mpc_kw.get("w_state", W_STATE)], tensors)), "optistate_kf_closed_loop")
        return (xs, fs, mst, fst, pws) if return_p_world else (xs, fs, mst, fst)
    # dense noise or a non-symmetric P0 (the joint filter step), or a caller-owned WarmStart: stepped from here
    if mpc_kw.get("warm", None) in (True, None) and "warm" in mpc_kw:
        del mpc_kw["warm"]
    if mpc_kw.get("warm", None) is False:
        mpc_kw["warm"] = None
    for t in range(T):
        forces, st = mpc_forces(x, body_ref[t], p[t], contact[t], **model, **mpc_kw)
        fs[t], mst[t] = forces[0], st
        res = kf_batch(imu[t:t + 1], p[t:t + 1], dp[t:t + 1], contact[t:t + 1], forces[0:1], x0=x, P0=Pm, Q=q_t, R=r_t, n_traj=N,
                       cov_model="mpc", body_ref=body_ref[t, 0:1], outputs=outputs, algo=algo, q_kind=q_kind, r_kind=r_kind,
                       p0_kind=p_kind, p0_is_symmetric=p_sym, **model)
        # the fed-back covariance: dense per trajectory; symmetric by construction on the packed-symmetric path
        x, Pm, p_kind = res.x_final, res.P_final, nv.MAT_DENSE_PER
        xs[t] = x
        if return_p_world:
            pws[t] = res.p_world_steps[0]
        fst |= res.status
    return (xs, fs, mst, fst, pws) if return_p_world else (xs, fs, mst, fst)
