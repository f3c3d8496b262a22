"""Batched entry point: filters N independent trajectories over T steps in one kernel launch.

This is the new call the reference does not have; per trajectory and per step it computes exactly what the
reference driver computes with
    KF.set_measurements(imu, KF.get_odom(p, dp, contact, imu)); KF.predict(p, f); KF.update()
(/root/reference/kalman_filter/kalman_filter.py:79-138,164-174; loop shape of
/root/reference/data_collection/data_conversion_Kalman_to_Training.py:193-201).

Layouts are structure-of-arrays with the trajectory / stream index fastest-varying (coalesced on the device):
per-step inputs [T, C, S], per-step outputs [T, C, N], per-trajectory arrays [C, N].  Trajectory i reads base
stream `stream_index[i]`, or `(i + stream_offset) % S` when no index is given, so thousands of Monte-Carlo members
can share a few input streams.
"""
from __future__ import annotations

import inspect
import warnings
from dataclasses import dataclass, field
from typing import Dict, Iterable, Optional

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _native as nv
from .settings import INITIAL_PARAMS

_OUT_ALIASES = {"p_trace": "p_trace_steps", "k_gain": "k_gain_steps", "p_checkpoints": "P_ckpt", "nis": "nis_steps"}
_OUT_SHAPES = {
    "x_steps": lambda T, N, K: (T, 12, N), "x_model_steps": lambda T, N, K: (T, 12, N),
    "p_world_steps": lambda T, N, K: (T, 12, N), "z_steps": lambda T, N, K: (T, 10, N),
    "p_trace_steps": lambda T, N, K: (T, N), "k_gain_steps": lambda T, N, K: (T, N), "nis_steps": lambda T, N, K: (T, N),
    "P_ckpt": lambda T, N, K: (K, 144, N), "x_final": lambda T, N, K: (12, N), "P_final": lambda T, N, K: (144, N),
    "K_final": lambda T, N, K: (120, N), "summary": lambda T, N, K: (nv.SUMMARY_ROWS, N),
}
_ALGOS = {"auto": nv.ALGO_AUTO, "joint": nv.ALGO_JOINT, "sequential": nv.ALGO_SEQUENTIAL}
_ALGO_NAMES = {nv.ALGO_JOINT: "joint", nv.ALGO_SEQUENTIAL: "sequential"}

# decoupled groups of the predict() model (include/optistate_kf.h OPTI_KF_FLAG_*): {th, w}, {x, vx}, {y, vy}, {z, vz}
_GROUP = torch.tensor([0, 0, 0, 1, 2, 3, 0, 0, 0, 1, 2, 3])
_CROSS_GROUP = _GROUP[:, None] != _GROUP[None, :]

SUMMARY_FIELDS = {
    "x_final": slice(0, 12), "p_diag": slice(12, 24), "rmse_truth": slice(24, 36), "rms_dev_nominal": slice(36, 48),
    "mean_nis": 48, "p_trace": 49, "k_gain": 50, "max_nis_sqrt": 51,
}


@dataclass
class KfBatchResult:
    """Device tensors of one kf_batch call.  `status[i]` is a bit mask (see optistate_kf.h OPTI_KF_ST_*)."""
    algo: str
    n_traj: int
    n_steps: int
    tensors: Dict[str, torch.Tensor] = field(default_factory=dict)
    status: Optional[torch.Tensor] = None

    def __getattr__(self, name):
        t = self.__dict__.get("tensors", {})
        if name in t:
            return t[name]
        raise AttributeError(name)

    def P_matrix(self, which: str = "P_final") -> torch.Tensor:
        """[..., 144, N] -> [..., N, 12, 12]."""
        t = self.tensors[which]
        return t.movedim(-1, -2).reshape(*t.shape[:-2], t.shape[-1], 12, 12)

    def summary_field(self, name: str) -> torch.Tensor:
        return self.tensors["summary"][SUMMARY_FIELDS[name]]


def _as_device(a, dtype, device, non_blocking=True):
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        t = a
    else:
        t = torch.from_numpy(np.ascontiguousarray(a))
    if t.device != device or t.dtype != dtype:
        t = t.to(device=device, dtype=dtype, non_blocking=non_blocking)
    return t.contiguous()


def _stream_tensor(a, C, name, dtype, device):
    t = _as_device(a, dtype, device)
    if t is None:
        return None, None, None
    if t.dim() == 2:
        t = t.unsqueeze(-1)
    if t.dim() != 3 or t.shape[1] != C:
        raise ValueError(f"{name} must have shape [T, {C}, S], got {tuple(t.shape)}")
    return t.contiguous(), t.shape[0], t.shape[2]


def _checked_stream_index(stream_index, N: int, S: int, device) -> torch.Tensor:
    """The kernels use the entries as gather offsets, so they are range-checked here (one small reduction; the gather path is not
    the streamed hot path)."""
    t = _as_device(stream_index, torch.int32, device).reshape(N)
    if N > 0:
        lo, hi = (int(v) for v in torch.aminmax(t))
        if lo < 0 or hi >= S:
            raise ValueError(f"stream_index entries must lie in [0, {S}), got [{lo}, {hi}]")
    return t


def _is_diagonal(m: torch.Tensor) -> bool:
    return bool(torch.count_nonzero(m - torch.diag(torch.diagonal(m))) == 0)


def _noise(a, n, N, name, dtype, device, kind=None):
    """Classifies a noise / covariance argument -> (tensor, kind).  Shapes: [n] shared diagonal, [n, N] diagonal per
    trajectory, [n, n] shared dense, [n*n, N] or [n, n, N] dense per trajectory.  A shared dense matrix that is
    exactly diagonal (np.diag(...), as the reference builds them) is passed on as a diagonal."""
    t = _as_device(a, dtype, device)
    shp = tuple(t.shape)
    if kind is None:
        if shp == (n,):
            kind = nv.MAT_DIAG
        elif shp == (n, n):  # also the [n, N] layout when N == n: pass kind= to disambiguate
            kind = nv.MAT_DENSE
        elif shp == (n, N):
            kind = nv.MAT_DIAG_PER
        elif shp in ((n * n, N), (n, n, N)):
            kind = nv.MAT_DENSE_PER
        else:
            raise ValueError(f"{name}: unsupported shape {shp} for n={n}, N={N}")
    if kind == nv.MAT_DENSE and _is_diagonal(t.reshape(n, n)):
        t, kind = torch.diagonal(t.reshape(n, n)).contiguous(), nv.MAT_DIAG
    return t.contiguous(), kind


def kf_batch(
    imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *,
    n_traj: Optional[int] = None, dtype: torch.dtype = torch.float64, stream_index=None, stream_offset: int = 0,
    outputs: Iterable[str] = ("x_steps",), ckpt_every: int = 0, truth=None, nominal=None, body_ref=None, z=None,
    algo: str = "auto", cov_model: str = "predict", q_kind=None, r_kind=None, p0_kind=None,
    dt: float = INITIAL_PARAMS.DT_mpc, mass: float = INITIAL_PARAMS.ROBOT_MASS, inertia=None,
    gravity: float = INITIAL_PARAMS.GRAVITY, device=None, out: Optional[Dict[str, torch.Tensor]] = None,
    summary_peers=None, p0_is_symmetric: Optional[bool] = None, structure: str = "auto", packed: bool = True,
) -> KfBatchResult:
    """Runs the Kalman filter over N trajectories x T steps on the current CUDA device.

    imu [T,6,S], p [T,12,S], dp [T,12,S], contact [T,4,S], f [T,12,S]: base input streams (torch CUDA tensors are
    used in place; NumPy arrays / CPU tensors are copied to the device).  `z` [T,10,S] may be given instead of
    imu/dp/contact (pre-formed measurements, see kf_measure).
    x0: [12] or [12,N] (default STARTING_STATE);  Q, R: see _noise (defaults INITIAL_PARAMS);  P0: None = Q.
    outputs: any of x_steps, x_model_steps, p_world_steps, z_steps, p_trace_steps (alias p_trace), k_gain_steps
    (k_gain), nis_steps, P_ckpt (p_checkpoints, needs ckpt_every), x_final, P_final, final (= both), K_final, summary.
    algo: "auto" | "sequential" | "joint" (see include/optistate_kf.h).  cov_model: "predict" | "mpc".
    out: optional preallocated output tensors by canonical name, and "workspace" (uint8 scratch of the streamed sequential
    path); a workspace that is missing or smaller than the library asks for is replaced in `out` by one of the queried size.
    p0_is_symmetric: skips the (synchronising) symmetry test of a dense P0 when the caller knows the answer, e.g. when P0
    is the P_final of a previous sequential call.
    structure: "auto" | "full" - the sequential kernels exploit that predict()'s F_d only couples attitude with body rate
    and each position with the velocity of its axis, so with a P0 without entries across those groups (None, diagonal, or
    a dense P0 whose cross-group entries are all zero - checked here) the cross-group entries of P are exact zeros at every
    step, in the reference too, and are neither stored nor multiplied (bit-identical results, less than half the
    arithmetic).  "full" keeps all 78 packed entries regardless (tests, comparison).
    packed: FP32 only - False keeps one trajectory per thread where the packed two-per-thread kernel (FFMA2) would be chosen.
    summary_peers: an optistate_b200.peer.PeerSummary - the summary is then written into this rank's columns of the
    job-wide [52, n_total] array on EVERY GPU of the box by the filter kernel itself (fused all-gather over NVLink peer
    stores); `result.summary` is the local column block, `summary_peers.tensor` the gathered array once
    `summary_peers.wait()` has run.
    """
    call = _filter_call(imu, p, dp, contact, f, x0, P0, Q, R, n_traj=n_traj, dtype=dtype, stream_index=stream_index,
                        stream_offset=stream_offset, outputs=outputs, ckpt_every=ckpt_every, truth=truth, nominal=nominal,
                        body_ref=body_ref, z=z, algo=algo, cov_model=cov_model, q_kind=q_kind, r_kind=r_kind, p0_kind=p0_kind, dt=dt,
                        mass=mass, inertia=inertia, gravity=gravity, device=device, out=out, summary_peers=summary_peers,
                        p0_is_symmetric=p0_is_symmetric, structure=structure, packed=packed)
    with torch.cuda.device(call.device):
        _attach_workspace(call, out)
        nv.check(int(call.ext.kf_batch(call.cfg, call.consts, call.tensors)), "optistate_kf_batch")
    return call.result(summary_peers)


@dataclass
class _FilterCall:
    """The prepared arguments of one filter run (kf_batch, and the forward pass of kf_smooth)."""
    ext: object
    device: torch.device
    cfg: dict
    consts: dict
    tensors: Dict[str, torch.Tensor]
    want: list
    status: torch.Tensor
    n_traj: int
    n_steps: int

    def result(self, summary_peers=None, extra=()) -> KfBatchResult:
        res = {k: self.tensors[k] for k in (*self.want, *extra)}
        if summary_peers is not None and "summary" in res:
            res["summary"] = summary_peers.local
        return KfBatchResult(algo=_ALGO_NAMES[self.cfg["algo"]], n_traj=self.n_traj, n_steps=self.n_steps, tensors=res, status=self.status)


def _out_tensor(out, name, shape, dtype, device) -> torch.Tensor:
    """The caller's out[name], which must be `shape` `dtype`, or a new tensor."""
    if out is not None and name in out:
        if tuple(out[name].shape) != shape or out[name].dtype != dtype:
            raise ValueError(f"out['{name}'] must be {shape} {dtype}")
        return out[name]
    return torch.empty(shape, dtype=dtype, device=device)


def _scratch(out, key, nbytes: int, device) -> torch.Tensor:
    """uint8 device scratch of at least nbytes (and at least 1): out[key] when large enough, else a new one kept in out[key] for
    the caller's next call with the same shapes."""
    t = out.get(key) if out is not None else None
    if t is None or t.numel() < nbytes:
        t = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        if out is not None:
            out[key] = t
    return t


def _attach_workspace(call: _FilterCall, out):
    """Scratch for the streamed SEQUENTIAL path (measurement pre-pass + TMA-fed kernel); 0 bytes when unused."""
    ws_bytes = call.ext.kf_batch(dict(call.cfg, query_workspace=1), call.consts, call.tensors)
    if ws_bytes < 0:
        nv.check(int(ws_bytes), "optistate_kf_workspace_bytes")
    if ws_bytes > 0:
        call.tensors["workspace"] = _scratch(out, "workspace", int(ws_bytes), call.device)


def _filter_call(imu, p, dp, contact, f, x0, P0, Q, R, *, n_traj, dtype, stream_index, stream_offset, outputs, ckpt_every, truth,
                 nominal, body_ref, z, algo, cov_model, q_kind, r_kind, p0_kind, dt, mass, inertia, gravity, device, out, summary_peers,
                 p0_is_symmetric, structure, packed) -> _FilterCall:
    """kf_batch's argument handling: inputs to the device, noise kinds, output tensors, the resolved algo."""
    nv.require_cuda()
    ext = nv.ext()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dtype not in (torch.float64, torch.float32):
        raise ValueError("dtype must be torch.float64 or torch.float32")

    tensors: Dict[str, torch.Tensor] = {}
    T = S = None
    for name, arr, C in (("imu", imu, 6), ("p", p, 12), ("dp", dp, 12), ("contact", contact, 4), ("f", f, 12),
                         ("z_in", z, 10), ("body_ref", body_ref, 12), ("truth", truth, 12), ("nominal", nominal, 12)):
        t, tT, tS = _stream_tensor(arr, C, name, dtype, device)
        if t is None:
            continue
        if T is None:
            T, S = tT, tS
        elif (tT, tS) != (T, S):
            raise ValueError(f"{name} has [T,S]=({tT},{tS}), expected ({T},{S})")
        tensors[name] = t
    if T is None:
        raise ValueError("no input streams given")
    N = int(S if n_traj is None else n_traj)
    phases = nv.PHASE_ALL if z is None else (nv.PHASE_PREDICT | nv.PHASE_UPDATE)

    x0_t = _as_device(INITIAL_PARAMS.STARTING_STATE.reshape(12) if x0 is None else x0, dtype, device)
    x0_t = x0_t.reshape(12) if x0_t.numel() == 12 else x0_t.reshape(12, N)
    tensors["x0"] = x0_t.contiguous()
    tensors["Q"], qk = _noise(INITIAL_PARAMS.Q if Q is None else Q, 12, N, "Q", dtype, device, q_kind)
    tensors["R"], rk = _noise(INITIAL_PARAMS.R if R is None else R, 10, N, "R", dtype, device, r_kind)
    pk = nv.MAT_NONE
    p0_symmetric = True
    if structure not in ("auto", "full"):
        raise ValueError("structure must be 'auto' or 'full'")
    flags = nv.FLAG_FULL_COVARIANCE if structure == "full" else 0
    if not packed:
        flags |= nv.FLAG_SCALAR_FP32
    if P0 is not None:
        tensors["P0"], pk = _noise(P0, 12, N, "P0", dtype, device, p0_kind)
        if pk in (nv.MAT_DENSE, nv.MAT_DENSE_PER):
            m = tensors["P0"].reshape(12, 12, -1)
            p0_symmetric = bool(torch.equal(m, m.transpose(0, 1))) if p0_is_symmetric is None else bool(p0_is_symmetric)
            if structure == "auto" and p0_is_symmetric is None and p0_symmetric and cov_model != "mpc":
                # (the test synchronises, like the symmetry test; callers that pass p0_is_symmetric skip both)
                if not bool(torch.count_nonzero(m[_CROSS_GROUP.to(device)])):
                    flags |= nv.FLAG_P0_DECOUPLED
    if stream_index is not None:
        tensors["stream_index"] = _checked_stream_index(stream_index, N, S, device)

    want = []
    for o in outputs:
        o = _OUT_ALIASES.get(o, o)
        want.extend(["x_final", "P_final"] if o == "final" else [o])
    n_ckpt = T // ckpt_every if ckpt_every else 0
    for o in want:
        if o not in _OUT_SHAPES:
            raise ValueError(f"unknown output '{o}'")
        shape = _OUT_SHAPES[o](T, N, n_ckpt)
        if o == "summary" and summary_peers is not None:
            if summary_peers.dtype != dtype or summary_peers.n_local != N or summary_peers.device != device:
                raise ValueError("summary_peers was set up for another dtype, device or shard size")
            tensors[o] = summary_peers.tensor
        else:
            tensors[o] = _out_tensor(out, o, shape, dtype, device)
    status = out["status"] if out is not None and "status" in out else torch.zeros(N, dtype=torch.int32, device=device)
    tensors["status"] = status

    cfg = dict(dtype=nv.F64 if dtype == torch.float64 else nv.F32, algo=_ALGOS[algo],
               cov_model=nv.COV_MPC if cov_model == "mpc" else nv.COV_PREDICT, phases=phases, n_traj=N, n_steps=T,
               n_streams=S, stream_offset=int(stream_offset), x0_per_traj=int(x0_t.dim() == 2), p0_kind=pk, q_kind=qk,
               r_kind=rk, ckpt_every=int(ckpt_every), want_K=int("K_final" in want), flags=flags)
    if summary_peers is not None and "summary" in want:
        cfg.update(summary_peers.cfg())
    if cfg["algo"] == nv.ALGO_AUTO:
        # a symmetric dense P0 is fine for the packed-symmetric kernel; a non-symmetric one needs the joint form
        probe = dict(cfg, algo=nv.ALGO_SEQUENTIAL)
        cfg["algo"] = nv.ALGO_SEQUENTIAL if (p0_symmetric and ext.kf_resolve_algo(probe) == nv.ALGO_SEQUENTIAL) else nv.ALGO_JOINT
    elif cfg["algo"] == nv.ALGO_SEQUENTIAL and not p0_symmetric:
        raise ValueError("algo='sequential' needs a symmetric P0")
    inertia = np.diag(INITIAL_PARAMS.INERTIA_ROT) if inertia is None else np.asarray(inertia, float).reshape(3)
    consts = dict(dt=float(dt), mass=float(mass), inertia0=float(inertia[0]), inertia1=float(inertia[1]),
                  inertia2=float(inertia[2]), gravity=float(gravity))
    return _FilterCall(ext=ext, device=device, cfg=cfg, consts=consts, tensors=tensors, want=want, status=status, n_traj=N, n_steps=T)


_SMOOTH_OUTPUTS = ("x_smooth", "var_smooth")
EM_STATS_ROWS = 23
EM_FIELDS = {"Sw": slice(0, 12), "Sv": slice(12, 22), "loglik": 22}
_FILTER_SIGNATURE = inspect.signature(kf_batch)


@dataclass(frozen=True)
class _Backward:
    """One of the five backward passes over the sequential filter (include/optistate_kf.h)."""
    who: str        # public name, in ValueErrors
    entry: str      # binding; with cfg query_storage = 1 it returns the storage size instead of running
    storage: str    # key of the library's scratch in `out`
    c_run: str      # C entry and storage query, in nv.check messages
    c_storage: str
    full: bool      # the full-covariance kernel: either covariance model, any symmetric P0 (_filter_call refuses others)
    stats: bool     # the E-step: noise_stats out, x_smooth optional
    adj: bool = False  # the adjoint: x_bar in, grad out, no smoothed outputs


_KF_SMOOTH = _Backward("kf_smooth", "kf_smooth", "smooth_storage", "optistate_kf_smooth",
                       "optistate_kf_smooth_storage_bytes", False, False)
_KF_SMOOTH_FULL = _Backward("kf_smooth_full", "kf_smooth_full", "smooth_storage", "optistate_kf_smooth_full",
                            "optistate_kf_smooth_full_storage_bytes", True, False)
_KF_NOISE_STATS = _Backward("kf_noise_stats", "kf_noise_em_stats", "em_storage", "optistate_kf_noise_em_stats",
                            "optistate_kf_noise_em_storage_bytes", False, True)
_KF_NOISE_STATS_FULL = _Backward("kf_noise_stats_full", "kf_noise_em_full_stats", "em_storage", "optistate_kf_noise_em_full_stats",
                                 "optistate_kf_noise_em_full_storage_bytes", True, True)
_KF_VJP = _Backward("kf_vjp", "kf_adjoint", "adj_storage", "optistate_kf_adjoint", "optistate_kf_adjoint_storage_bytes", False, False,
                    adj=True)
ADJ_ROWS = 46
ADJ_FIELDS = {"Q": slice(0, 12), "R": slice(12, 22), "x0": slice(22, 34), "P0": slice(34, 46)}


def _backward_call(v: _Backward, args, outputs, kw):
    """The forward pass's _FilterCall (kf_batch's keywords and defaults) with what the backward kernel refuses refused here, and
    the remaining outputs; returns (call, kw bound to kf_batch's signature, the backward outputs asked for)."""
    try:
        bound = _FILTER_SIGNATURE.bind(*args, **kw)
    except TypeError as e:  # a keyword kf_batch does not take
        raise TypeError(f"{v.who}() {e}") from None
    bound.apply_defaults()
    kw = bound.arguments
    who, full = v.who, v.full
    if not full and kw["cov_model"] != "predict":
        raise ValueError(f"{who} supports the predict() covariance model only (predict_mpc makes F_d dense)")
    if not full and kw["structure"] != "auto":
        raise ValueError(f"{who} needs the decoupled-group form of P; structure='full' keeps cross-group entries")
    if kw["algo"] == "joint":
        raise ValueError(f"{who} runs on the sequential filter; algo='joint' is not supported")
    outputs = list(outputs)
    smooth_want = [o for o in outputs if o in _SMOOTH_OUTPUTS]
    if v.adj and smooth_want:
        raise ValueError(f"{who} has no smoothed outputs")
    if not v.stats and not v.adj and "x_smooth" not in smooth_want:
        smooth_want.insert(0, "x_smooth")
    kw.update(outputs=[o for o in outputs if o not in _SMOOTH_OUTPUTS], algo="sequential" if kw["algo"] == "auto" else kw["algo"])
    call = _filter_call(**kw)
    cfg = call.cfg
    if cfg["q_kind"] not in (nv.MAT_DIAG, nv.MAT_DIAG_PER) or cfg["r_kind"] not in (nv.MAT_DIAG, nv.MAT_DIAG_PER):
        raise ValueError(f"{who} needs diagonal Q and R " + ("(the sequential filter takes no dense noise)" if full else
                                                               "(dense noise couples the decoupled groups)"))
    if not full and cfg["p0_kind"] in (nv.MAT_DENSE, nv.MAT_DENSE_PER) and not cfg["flags"] & nv.FLAG_P0_DECOUPLED:
        raise ValueError(f"{who} needs a P0 without entries across the groups {{th, w}}, {{x, vx}}, {{y, vy}}, {{z, vz}}")
    return call, kw, smooth_want


def _run_backward(v: _Backward, args, outputs, kw, x_bar=None) -> KfBatchResult:
    """The forward pass of _backward_call, the smoothed outputs, noise_stats or the adjoint's x_bar and grad, and the library's
    storage attached, then the backward entry."""
    call, kw, smooth_want = _backward_call(v, args, outputs, kw)
    cfg = call.cfg
    T, N, out, dtype = call.n_steps, call.n_traj, kw["out"], kw["dtype"]
    for o in smooth_want:
        call.tensors[o] = _out_tensor(out, o, (T, 12, N), dtype, call.device)
    extra = smooth_want
    if v.stats:
        call.tensors["noise_stats"] = _out_tensor(out, "noise_stats", (EM_STATS_ROWS, N), dtype, call.device)
        extra = ["noise_stats", *smooth_want]
    if v.adj:
        xb = _as_device(x_bar, dtype, call.device)
        if tuple(xb.shape) != (T, 12, N):
            raise ValueError(f"{v.who}: grad_x_steps must have the shape of x_steps, {(T, 12, N)}, got {tuple(xb.shape)}")
        call.tensors["x_bar"] = xb
        call.tensors["grad"] = _out_tensor(out, "grad", (ADJ_ROWS, N), dtype, call.device)
        extra = ["grad"]
    entry = getattr(call.ext, v.entry)
    with torch.cuda.device(call.device):
        _attach_workspace(call, out)
        st_bytes = entry(dict(cfg, query_storage=1), call.consts, call.tensors)
        nv.check(int(min(st_bytes, 0)), v.c_storage)
        call.tensors[v.storage] = _scratch(out, v.storage, int(st_bytes), call.device)
        nv.check(int(entry(cfg, call.consts, call.tensors)), v.c_run)
    return call.result(kw["summary_peers"], extra=extra)


def kf_smooth(imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *, outputs: Iterable[str] = ("x_smooth",),
              **kw) -> KfBatchResult:
    """Fixed-interval Rauch-Tung-Striebel smoother: runs the filter exactly as kf_batch runs it with the same arguments, then a
    backward kernel that conditions every step's estimate on ALL measurements of the recording (offline use).  The keywords
    other than outputs are kf_batch's, with its defaults.

    outputs: x_smooth [T,12,N] (smoothed state, the default), var_smooth [T,12,N] (diagonal of the smoothed covariance), and any
    kf_batch output - those come from the same forward pass.  out: as for kf_batch, plus "smooth_storage" (uint8 scratch of
    optistate_kf_smooth_storage_bytes: the packed posterior covariance of every step, 240 B per trajectory-step in FP64, and the
    filter's x_steps / x_model_steps when they are not outputs), replaced in `out` when missing or too small.
    Supported: the sequential algo with the predict() covariance model, diagonal Q and R and a P0 without entries across the
    groups {th, w}, {x, vx}, {y, vy}, {z, vz}; anything else raises ValueError.  status gains OPTI_KF_ST_SMOOTH_NOT_PD (32).
    """
    return _run_backward(_KF_SMOOTH, (imu, p, dp, contact, f, x0, P0, Q, R), outputs, kw)


def kf_smooth_full(imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *, outputs: Iterable[str] = ("x_smooth",),
                   **kw) -> KfBatchResult:
    """The fixed-interval smoother of kf_smooth on the FULL 12x12 covariance (DESIGN.md section 0.2): for the predict_mpc
    covariance model (cov_model="mpc", whose element-wise F_d = exp(dt F) makes P dense) and for a P0 with entries across the
    groups, which kf_smooth refuses.  Arguments (the keywords other than outputs are kf_batch's), outputs (x_smooth, var_smooth
    and any kf_batch output) and out["smooth_storage"] as for kf_smooth; the storage holds all 78 entries of P+ per step (624 B
    per trajectory-step in FP64).  The forward pass runs the sequential filter's full-covariance kernels, whose outputs equal
    kf_batch's with the same arguments.

    The closed loop's output, smoothed offline:

        xs, fs, *_ = estimate_state_mpc_batch(...)
        res = kf_smooth_full(imu, p, dp, contact, fs, x0, P0, Q, R, cov_model="mpc", body_ref=body_ref[:, 0], n_traj=N)

    Raises ValueError for algo="joint", dense Q or R, and a non-symmetric P0.  FP64 is the dtype for real data: under the
    predict_mpc model with identified noise P- reaches condition numbers near 1e8, which FP32 cannot resolve.
    status gains OPTI_KF_ST_SMOOTH_NOT_PD (32).
    """
    return _run_backward(_KF_SMOOTH_FULL, (imu, p, dp, contact, f, x0, P0, Q, R), outputs, kw)


def kf_noise_stats(imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *, outputs: Iterable[str] = (),
                   **kw) -> KfBatchResult:
    """E-step of expectation-maximisation for diagonal Q and R (DESIGN.md section 0): runs the filter and the smoother's backward
    kernel exactly as kf_smooth does with the same arguments, and returns `noise_stats` [23, N] per trajectory:
        rows 0-11   Sw = sum_t E[w_t^2 | Z]   over the T transitions t = -1 .. T-2 (x_{-1} ~ N(x0, P0), P0 = Q when None)
        rows 12-21  Sv = sum_t E[v_t^2 | Z]   over the T measurements
        row 22      the prediction-error log-likelihood sum_t log N(z_t; H x-_t, H P-_t H^T + R) of the filter that ran
    The M-step is Q = diag(Sw) / T, R = diag(Sv) / T (kf_noise_em).  The keywords other than outputs are kf_batch's, with its
    defaults.  outputs: x_smooth, var_smooth and any kf_batch output, all optional.  out: as for kf_smooth, with "noise_stats" and
    "em_storage" (uint8 scratch of optistate_kf_noise_em_storage_bytes).  Refuses what kf_smooth refuses, with the same ValueErrors.
    """
    return _run_backward(_KF_NOISE_STATS, (imu, p, dp, contact, f, x0, P0, Q, R), outputs, kw)


def kf_noise_stats_full(imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *, outputs: Iterable[str] = (),
                        **kw) -> KfBatchResult:
    """The E-step of kf_noise_stats on the FULL covariance (DESIGN.md section 0.3): the forward pass and backward kernel of
    kf_smooth_full, so the predict_mpc covariance model (cov_model="mpc", with body_ref) and a coupled or dense symmetric P0 are
    taken.  The keywords other than outputs are kf_batch's, with its defaults.  Returns `noise_stats` [23, N] with the rows of
    kf_noise_stats (the innovation covariance of the log-likelihood is the dense H P- H^T + R), and x_smooth / var_smooth or any
    kf_batch output when asked for.  out: as for kf_smooth_full, with "noise_stats" and "em_storage"
    (optistate_kf_noise_em_full_storage_bytes).  Refuses what kf_smooth_full refuses: algo="joint", dense Q or R and a
    non-symmetric P0 raise ValueError.
    """
    return _run_backward(_KF_NOISE_STATS_FULL, (imu, p, dp, contact, f, x0, P0, Q, R), outputs, kw)


def kf_vjp(imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *, grad_x_steps, outputs: Iterable[str] = (),
           **kw) -> KfBatchResult:
    """Gradient of the filter's x_steps (DESIGN.md section 0.4): runs the filter exactly as kf_batch runs it with the same
    arguments, then an adjoint kernel backwards over it, and returns `grad` [46, N] per trajectory, for any loss L with
    dL/dx_steps = grad_x_steps [T, 12, N]:
        rows 0-11   dL/dQ_ii through the predicted covariances (not through P0 = Q: add rows 34-45 when P0 is None)
        rows 12-21  dL/dR_kk
        rows 22-33  dL/dx0
        rows 34-45  the diagonal of dL/dP0 (of the initial covariance, Q when P0 is None)
    The keywords other than grad_x_steps and outputs are kf_batch's, with its defaults; outputs: any kf_batch output, from the same
    forward pass.  out: as for kf_batch, plus "grad" and "adj_storage" (uint8 scratch of optistate_kf_adjoint_storage_bytes: the
    smoother's storage, the measurements and the leg moments of the mean model).  At an exactly axis-aligned attitude (e.g. the
    all-zero start) the mean model's trunc(R^T) jumps and the gradient is the almost-everywhere one.  Refuses what kf_smooth
    refuses, with the same ValueErrors; a dense P0 without cross-group entries is taken, rows 34-45 then hold its diagonal only.
    """
    return _run_backward(_KF_VJP, (imu, p, dp, contact, f, x0, P0, Q, R), outputs, kw, x_bar=grad_x_steps)


def _grad_like(g: torch.Tensor, inp: torch.Tensor, per_traj: bool, n: int) -> torch.Tensor:
    """A per-trajectory gradient g [n, N] in the shape of the input it belongs to, by the kind the forward pass resolved for it:
    per trajectory ([n, N]) as it is, shared ([n], or a diagonal [n, n]) summed over the trajectories."""
    if per_traj:
        out = g
    else:
        out = g.sum(dim=1)
        if inp.numel() != n:
            out = torch.diag(out)
    return out.to(dtype=inp.dtype, device=inp.device).reshape(inp.shape)


class _KfStates(torch.autograd.Function):
    @staticmethod
    def forward(ctx, kw, imu, p, dp, contact, f, x0, P0, Q, R):
        args = (imu, p, dp, contact, f, x0, P0, Q, R)
        call, _, _ = _backward_call(_KF_VJP, tuple(a.detach() if isinstance(a, torch.Tensor) else a for a in args), ("x_steps",), kw)
        cfg = call.cfg
        if ctx.needs_input_grad[7] and cfg["p0_kind"] in (nv.MAT_DENSE, nv.MAT_DENSE_PER):
            raise ValueError("kf_states: a dense P0 cannot require grad (the adjoint returns the diagonal of dL/dP0 only)")
        with torch.cuda.device(call.device):
            _attach_workspace(call, kw.get("out"))
            nv.check(int(call.ext.kf_batch(call.cfg, call.consts, call.tensors)), "optistate_kf_batch")
        # the backward pass re-runs the filter from these inputs: saved through autograd, an input changed in place in between
        # raises instead of giving the gradient at other values
        kw_t = sorted(k for k, v in kw.items() if isinstance(v, torch.Tensor))
        arg_t = [k for k, a in enumerate(args) if isinstance(a, torch.Tensor)]
        ctx.save_for_backward(*(args[k] for k in arg_t), *(kw[k] for k in kw_t))
        ctx.layout = arg_t, kw_t
        ctx.args = tuple(None if isinstance(a, torch.Tensor) else a for a in args)
        ctx.kw = {k: v for k, v in kw.items() if k not in kw_t}
        # the kinds the forward pass resolved decide the gradients' shapes (a shape alone is ambiguous when N equals n)
        ctx.per_traj = dict(Q=cfg["q_kind"] == nv.MAT_DIAG_PER, R=cfg["r_kind"] == nv.MAT_DIAG_PER, P0=cfg["p0_kind"] == nv.MAT_DIAG_PER,
                            x0=bool(cfg["x0_per_traj"]))
        return call.tensors["x_steps"]

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        arg_t, kw_t = ctx.layout
        saved = ctx.saved_tensors
        args = list(ctx.args)
        for j, k in enumerate(arg_t):
            args[k] = saved[j]
        kw = dict(ctx.kw, **{k: saved[len(arg_t) + j] for j, k in enumerate(kw_t)})
        x0, P0, Q, R = args[5:]
        res = kf_vjp(*args, grad_x_steps=g.contiguous(), **kw)
        bad = res.status[res.status != 0]
        if bad.numel():
            bits = int(np.bitwise_or.reduce(np.unique(bad.cpu().numpy())))
            warnings.warn(f"kf_states: {bad.numel()} trajectories have a non-zero status (bits {bits:#x}, include/optistate_kf.h "
                          "OPTI_KF_ST_*): their gradients come from a filter or adjoint pivot that was not positive and finite, or "
                          "from a step without a stance leg", RuntimeWarning, stacklevel=2)
        grad = res.grad
        need = ctx.needs_input_grad
        gq = grad[ADJ_FIELDS["Q"]]
        if P0 is None:
            gq = gq + grad[ADJ_FIELDS["P0"]]
        out = [None] * 10
        per = ctx.per_traj
        if need[6]:
            out[6] = _grad_like(grad[ADJ_FIELDS["x0"]], x0, per["x0"], 12)
        if need[7]:
            out[7] = _grad_like(grad[ADJ_FIELDS["P0"]], P0, per["P0"], 12)
        if need[8]:
            out[8] = _grad_like(gq, Q, per["Q"], 12)
        if need[9]:
            out[9] = _grad_like(grad[ADJ_FIELDS["R"]], R, per["R"], 10)
        return tuple(out)


def kf_states(imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, **kw) -> torch.Tensor:
    """kf_batch's x_steps [T, 12, N] as a differentiable function of Q, R, x0 and P0: gradients of any loss on it reach the
    filter's parameters through torch autograd, whose backward runs kf_vjp (the forward pass again, then the adjoint kernel; no
    storage is held between the two).  The keywords are kf_batch's other than outputs.  Gradients come back in each input's own
    shape: Q, R and P0 diagonal ([n] or a diagonal [n, n] shared - summed over the trajectories - or [n, N]), x0 [12] or [12, N].
    With P0 None the initial covariance is Q, and its gradient is added to Q's.  Refuses what kf_smooth refuses, and a dense P0
    that requires grad (the adjoint returns the diagonal of dL/dP0 only), with ValueErrors.  Sensor streams get no gradient.
    The backward pass re-runs the filter from the saved inputs: one changed in place in between makes autograd raise.  It reads
    the status words of that filter run and of the adjoint (one host synchronisation) and warns (RuntimeWarning) when a
    trajectory's is non-zero - a pivot that was not positive and finite, or a step without a stance leg - since its gradient is
    then not to be trusted; kf_vjp returns the status words themselves.  The result is differentiable once.

        q = torch.log(torch.tensor(Q0, device="cuda")).requires_grad_()
        loss = ((kf_states(imu, p, dp, contact, f, Q=q.exp(), n_traj=N) - truth_steps) ** 2).mean()
        loss.backward()  # q.grad
    """
    if "outputs" in kw:
        raise TypeError("kf_states() returns x_steps; it takes no outputs")
    return _KfStates.apply(dict(kw), imu, p, dp, contact, f, x0, P0, Q, R)


@dataclass
class KfNoiseEmResult:
    """Result of kf_noise_em.  Q [12, N] / R [10, N] (or [12] / [10] with shared=True) are the estimates after the last M-step;
    loglik[k] is the log-likelihood of every trajectory under the k-th iterate (the E-step of iteration k), so the last row
    belongs to the iterate before Q, R.  status: the OR of the filter's status words over all iterations."""
    Q: torch.Tensor
    R: torch.Tensor
    loglik: torch.Tensor
    iterations: int
    converged: bool
    status: torch.Tensor


def kf_noise_em(
    imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *, iters: int = 50, tol: Optional[float] = None,
    shared: bool = False, n_traj: Optional[int] = None, dtype: torch.dtype = torch.float64, stream_index=None,
    stream_offset: int = 0, z=None, dt: float = INITIAL_PARAMS.DT_mpc, mass: float = INITIAL_PARAMS.ROBOT_MASS, inertia=None,
    gravity: float = INITIAL_PARAMS.GRAVITY, device=None, out: Optional[Dict[str, torch.Tensor]] = None,
) -> KfNoiseEmResult:
    """Maximum-likelihood diagonal Q and R from the sensor streams alone, by expectation-maximisation: each iteration runs
    kf_noise_stats (filter, smoother, E-step) with the current Q, R and sets Q = Sw / T, R = Sv / T - per trajectory, or with
    shared=True pooled over all trajectories (sums over N T).  The M-step runs as torch ops on the device.

    Q, R: the start, diagonal ([12] / [10], [12, N] / [10, N], or a diagonal matrix; default settings.py's).  P0 stays what the
    caller passes for every iteration; None holds it at the starting Q.  The filter is re-linearised each iteration (F and x-
    follow the new estimates), so the log-likelihood is not guaranteed to rise, though it does on typical recordings.
    Known limitation (DESIGN.md section 0): q of x and y is unobservable and stays at its start, and the estimates describe the
    affine model the filter runs, whose attitude rows use R^T rather than the mean model's trunc(R^T).
    tol: stop once the largest relative increase of the log-likelihood (per trajectory; pooled with shared=True) falls below
    it - one host synchronisation per iteration, only when tol is given.  Storage and workspace are reused across iterations.
    """
    return _noise_em("kf_noise_em", kf_noise_stats, (imu, p, dp, contact, f, x0, P0, Q, R), dict(
        n_traj=n_traj, dtype=dtype, stream_index=stream_index, stream_offset=stream_offset, z=z, dt=dt, mass=mass, inertia=inertia,
        gravity=gravity, device=device, out=out), iters, tol, shared)


def kf_noise_em_full(
    imu, p, dp, contact, f, x0=None, P0=None, Q=None, R=None, *, iters: int = 50, tol: Optional[float] = None,
    shared: bool = False, n_traj: Optional[int] = None, dtype: torch.dtype = torch.float64, stream_index=None,
    stream_offset: int = 0, z=None, cov_model: str = "predict", body_ref=None, dt: float = INITIAL_PARAMS.DT_mpc,
    mass: float = INITIAL_PARAMS.ROBOT_MASS, inertia=None, gravity: float = INITIAL_PARAMS.GRAVITY, device=None,
    out: Optional[Dict[str, torch.Tensor]] = None,
) -> KfNoiseEmResult:
    """kf_noise_em on the FULL covariance (DESIGN.md section 0.3): each iteration runs kf_noise_stats_full, so the filter may be
    the predict_mpc covariance model the reference's conversion driver runs (cov_model="mpc", body_ref [T, 12, S]: its rows 0-2 are
    the reference body angles of every step), and P0 may be coupled or dense (symmetric).  Arguments, M-step, tol and result as
    for kf_noise_em; P0 is held at the caller's value (or at the starting Q) across iterations.

    Q and R of the closed loop's filter, from the sensor streams alone:

        xs, fs, *_ = estimate_state_mpc_batch(imu, p, dp, contact, ref)
        em = kf_noise_em_full(imu, p, dp, contact, fs, cov_model="mpc", body_ref=ref[:, 0], n_traj=N, shared=True)

    The forces fs are inputs here and stay fixed across iterations: with a new Q and R the closed loop would compute other forces,
    and EM does not re-run it.  The estimate is the noise of the affine model the filter runs (DESIGN.md section 0.1's caveat), and
    under predict_mpc that model is further from the mean model: F_d = 1 1^T + D is not the mean model's Jacobian, so Q absorbs
    the difference and is not the process noise of the robot.  FP64 is the dtype for real data (kf_smooth_full).
    """
    return _noise_em("kf_noise_em_full", kf_noise_stats_full, (imu, p, dp, contact, f, x0, P0, Q, R), dict(
        n_traj=n_traj, dtype=dtype, stream_index=stream_index, stream_offset=stream_offset, z=z, cov_model=cov_model,
        body_ref=body_ref, dt=dt, mass=mass, inertia=inertia, gravity=gravity, device=device, out=out), iters, tol, shared)


def _noise_em(who, stats_fn, args, filter_kw, iters, tol, shared) -> KfNoiseEmResult:
    """The EM loop of kf_noise_em / kf_noise_em_full around the E-step stats_fn, which gets the filter's arguments args
    (imu .. R) and keywords filter_kw with the current Q, R and P0."""
    if iters < 1:
        raise ValueError("iters must be >= 1")
    nv.require_cuda()
    imu, p, dp, contact, f, x0, P0, Q, R = args
    n_traj, dtype, z = filter_kw["n_traj"], filter_kw["dtype"], filter_kw["z"]
    out = {} if filter_kw["out"] is None else filter_kw["out"]  # storage and workspace of the first E-step, reused by the others
    device = torch.device("cuda", torch.cuda.current_device()) if filter_kw["device"] is None else torch.device(filter_kw["device"])
    base = z if z is not None else imu
    T, S = int(base.shape[0]), int(base.shape[2]) if base.ndim == 3 else 1
    N = int(S if n_traj is None else n_traj)

    def diag_start(a, default, n):
        t = _as_device(default if a is None else a, dtype, device)
        if t.shape == (n, n):
            if not _is_diagonal(t):
                raise ValueError(f"{who} estimates diagonal noise: Q and R must be diagonal")
            t = torch.diagonal(t)
        if t.shape == (n,):
            return t.clone() if shared else t[:, None].expand(n, N).contiguous()
        if t.shape != (n, N):
            raise ValueError(f"{who}: a noise start of shape {tuple(t.shape)} is not [{n}], [{n}, {n}] or [{n}, {N}]")
        if shared:
            raise ValueError(f"{who}: shared=True needs a shared start ([n] or a diagonal matrix)")
        return t.clone()

    q = diag_start(Q, INITIAL_PARAMS.Q, 12)
    r = diag_start(R, INITIAL_PARAMS.R, 10)
    kind = nv.MAT_DIAG if shared else nv.MAT_DIAG_PER
    p0, p0_kind = (q.clone(), kind) if P0 is None else (P0, None)
    status = torch.zeros(N, dtype=torch.int32, device=device)
    kw = dict(filter_kw, n_traj=N, device=device, out=out, q_kind=kind, r_kind=kind, p0_kind=p0_kind)
    lls, converged, prev = [], False, None
    for it in range(iters):
        res = stats_fn(imu, p, dp, contact, f, x0, p0, q, r, **kw)
        st = res.noise_stats
        status |= res.status
        ll = st[EM_STATS_ROWS - 1].clone()
        lls.append(ll)
        if shared:
            q = st[0:12].sum(dim=1) / (N * T)
            r = st[12:22].sum(dim=1) / (N * T)
        else:
            q = st[0:12] / T
            r = st[12:22] / T
        if tol is not None and prev is not None:
            if shared:
                a, b = prev.sum(), ll.sum()
                rel = (b - a) / a.abs()
            else:
                rel = ((ll - prev) / prev.abs()).max()
            if float(rel) < tol:
                converged = True
                break
        prev = ll
    loglik = torch.stack(lls) if lls else torch.empty((0, N), dtype=dtype, device=device)
    return KfNoiseEmResult(Q=q, R=r, loglik=loglik, iterations=len(lls), converged=converged, status=status)


def kf_measure(imu, p, dp, contact, *, dtype: torch.dtype = torch.float64, device=None, want_odom: bool = False):
    """Batched get_odom + set_measurements (kalman_filter.py:79-117): returns z [T,10,S] (and odom [T,4,S], status [S])."""
    nv.require_cuda()
    ext = nv.ext()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    tensors = {}
    T = S = None
    for name, arr, C in (("imu", imu, 6), ("p", p, 12), ("dp", dp, 12), ("contact", contact, 4)):
        t, tT, tS = _stream_tensor(arr, C, name, dtype, device)
        if T is None:
            T, S = tT, tS
        elif (tT, tS) != (T, S):
            raise ValueError(f"{name} has [T,S]=({tT},{tS}), expected ({T},{S})")
        tensors[name] = t
    tensors["z"] = torch.empty((T, 10, S), dtype=dtype, device=device)
    if want_odom:
        tensors["odom"] = torch.empty((T, 4, S), dtype=dtype, device=device)
    tensors["status"] = torch.zeros(S, dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        nv.check(ext.kf_measure(nv.F64 if dtype == torch.float64 else nv.F32, T, S, tensors), "optistate_kf_measure")
    if want_odom:
        return tensors["z"], tensors["odom"], tensors["status"]
    return tensors["z"], tensors["status"]


def fma_peak(dtype: torch.dtype = torch.float64, fma_per_thread: int = 1 << 16):
    """Measured FMA issue peak of the current device: (FLOP/s, seconds of the timed launch)."""
    nv.require_cuda()
    return nv.ext().fma_peak(nv.F64 if dtype == torch.float64 else nv.F32, int(fma_per_thread))
