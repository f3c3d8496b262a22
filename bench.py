#!/usr/bin/env python
"""Headline benchmark: Kalman-filter trajectory-steps/sec on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dtype f64|f32]
                    [--traj-per-gpu M | --traj-total M] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (config.workload): the Monte-Carlo noise sweep of BASELINE.json configs[2]/[3] - trajectories x 1,000 steps over
1,024 shared synthetic base streams, per-member diagonal Q/R perturbations, outputs = per-trajectory summaries (final x,
diag P, RMSE vs the label stream, RMS deviation from the nominal member, mean NIS, ...) - in FP64 by default because the
north-star target is stated on the FP64 FMA roofline with 1e-9 parity (--dtype f32 gives configs[2] verbatim).
    default            1,048,576 trajectories PER GPU  ("scaling": "weak")
    --traj-total M     M trajectories in the whole job, contiguous M/N per rank ("scaling": "strong"); 16777216 is
                       BASELINE configs[3] as written
One "step" of the bench = one full pass of the hot path over that batch: measurement pre-pass + the filter kernel; when
N > 1 the all-gather of the summaries is fused into the filter kernel (NVLink peer stores, optistate_b200/peer.py;
--gather nccl runs the NCCL all-gather instead).

  value      whole-job trajectory-steps/s, inputs resident in HBM, timed with CUDA events, max over ranks
  e2e        same through the public host-buffer API (KfHostPipeline around kf_batch) with pinned HOST buffers: H2D of
             streams + per-member noise and D2H of the summaries inside the timed region
  roofline   FMA roofline of the dominant kernel: `frac` = flops the kernel EXECUTES (ncu opcode counts of its time loop,
             read from profiles/) x steps/s / FMA peak; `frac_algorithmic` = the SURVEY 8(d) figure of 6,800 flops per
             trajectory-step on the same denominator (can exceed 1: the kernel skips structural zeros)
  parity_sample  members of the TIMED batch compared with the C oracle after the timed region; the run fails if they differ
  cpu_baseline   the oracle's C port of the reference filter on this box's host cores (bounded sample), and the unmodified
             reference class itself (oracle/_ref) on 1 core and on all cores

--impl reference times the CPU arm (oracle C port, all host threads) on a bounded sample per step.
"""
from __future__ import annotations

import argparse
import ast
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_ALGORITHMIC = 6800.0  # SURVEY.md 8(d): per trajectory-step, reference operand order, structural zeros skipped
METRIC = "kf_trajectory_steps_per_sec"
UNIT = "trajectory-steps/s"
DEFAULT_SHAPE = (1 << 20, 1000, 1024)  # trajectories per launch, steps, base streams of the captured ncu profiles
FP64_TOL, FP32_TOL_X, FP32_TOL_P = 1e-9, 1e-4, 2e-4  # parity_sample limits (tests/parity.py; FP32 x bound x5 as in the full-size test)


# ---- executed flops and DRAM traffic of the dominant kernel: read from the committed ncu summaries -----------------------
def _opcode_flops(ops, lanes):
    """Flops per trajectory-step from the per-opcode executed-instruction counts of one loop trip (tools/ncu_hot.py):
    FMA = 2, MUL / ADD = 1, packed FP32 instructions carry two trajectories each (lanes = 2 for the F2 kernel)."""
    f64 = 2 * ops.get("DFMA", 0) + ops.get("DMUL", 0) + ops.get("DADD", 0)
    f32 = 2 * ops.get("FFMA", 0) + ops.get("FMUL", 0) + ops.get("FADD", 0)
    f32x2 = 2 * (2 * ops.get("FFMA2", 0) + ops.get("FMUL2", 0) + ops.get("FADD2", 0))
    n_fp = sum(ops.get(k, 0) for k in ("DFMA", "DMUL", "DADD", "FFMA", "FMUL", "FADD", "FFMA2", "FMUL2", "FADD2"))
    return (f64 + f32 + f32x2) / lanes, n_fp


def _parse_metrics(path):
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    out = {}
    for line in open(path):
        m = re.match(r"(\S+) \[(\S*)\] (\S+)\s*$", line)
        if m:
            try:
                out[m.group(1)] = float(m.group(3).replace(",", "")) * unit.get(m.group(2), 1.0)
            except ValueError:
                pass
    return out


def kernel_profile(dtype: str, structure: str = "auto", tags=("r2", "r1")):
    """The ncu summary of the dominant kernel for this dtype / covariance structure, newest round first:
    profiles/<tag>_ncu_bench_kernel_<dtype>[_full]_{hotloop,metrics}.txt.  Returns None when no capture of the instantiation
    that is being timed exists (the kernel name in the capture is checked: a stale file must not describe another kernel)."""
    want_block = structure != "full"
    for tag in tags:
        for suffix in (("",) if want_block else ("_full", "")):
            hot = os.path.join(ROOT, "profiles", f"{tag}_ncu_bench_kernel_{dtype}{suffix}_hotloop.txt")
            met = os.path.join(ROOT, "profiles", f"{tag}_ncu_bench_kernel_{dtype}{suffix}_metrics.txt")
            if not os.path.isfile(hot):
                continue
            lines = open(hot).read().splitlines()
            name = lines[0] if lines else ""
            args = re.search(r"kf_seq_tma_kernel<([^>]*)>", name)
            if not args:
                continue
            targs = [a.strip() for a in args.group(1).split(",")]
            is_block = len(targs) >= 5 and targs[4].endswith("1")
            if is_block != want_block or not targs[1].endswith("1") or not targs[2].endswith("0"):
                continue  # not the <summary, no per-step outputs> instantiation of this structure
            ops = next((ast.literal_eval(ln) for ln in lines if ln.startswith("{'")), None)
            if not ops:
                continue
            lanes = 2 if "F2" in targs[0] else 1
            flops, n_fp = _opcode_flops(ops, lanes)
            prof = {"flops_executed": flops, "fp_instructions_per_thread_step": n_fp, "instructions_per_thread_step": sum(ops.values()),
                    "lanes": lanes, "kernel": "kf_seq_tma_kernel<" + args.group(1) + ">", "source": os.path.relpath(hot, ROOT),
                    "traffic_bytes": None, "grid": None}
            if os.path.isfile(met):
                m = _parse_metrics(met)
                if "dram__bytes_read.sum" in m and "dram__bytes_write.sum" in m:
                    prof["traffic_bytes"] = m["dram__bytes_read.sum"] + m["dram__bytes_write.sum"]
                    prof["grid"] = int(m.get("launch__grid_size", 0)) or None
                    prof["fp_pipe_active_pct"] = m.get("sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active" if lanes == 1 and dtype == "f64"
                                                       else "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active")
                    prof["metrics_source"] = os.path.relpath(met, ROOT)
            return prof
    return None


def algorithmic_bytes(n_local, T, S, esz):
    """Algorithmic bytes of one launch: every base-stream channel read once (p, f, z, two label streams = 58 scalars per
    stream-step) + 22 noise scalars in and 52 summary scalars out per trajectory."""
    return (58 * T * S + (22 + 52) * n_local) * esz


DUMP_MEMBERS = 1 << 16  # --dump-outputs: 52 summary rows x 65,536 members x 8 B = 27 MB, under the 64 MB a dump may take


def dump_members(n: int) -> np.ndarray:
    """Member ids whose outputs --dump-outputs writes: all of them up to DUMP_MEMBERS, else a sorted sample drawn from a fixed
    seed, so that every run of the same shape writes the same members."""
    if n <= DUMP_MEMBERS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_MEMBERS, replace=False))


def dump_outputs(path: str, arrays: dict) -> None:
    os.makedirs(path, exist_ok=True)
    for name, arr in arrays.items():
        assert arr.dtype in (np.float32, np.float64), (name, arr.dtype)
        np.save(os.path.join(path, name + ".npy"), arr)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--traj-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--traj-total", type=int, default=0, help="strong scaling: trajectories of the whole job (16777216 = BASELINE configs[3])")
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--structure", default="auto", choices=["auto", "full"], help="full: carry all 78 packed covariance entries")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--e2e-upload", default="auto", choices=["auto", "shared", "shared-lowprio", "replicated"],
                    help="N > 1, e2e: every rank uploads all base streams (replicated), or 1/N of them + an NVLink all-gather on a "
                         "high-priority NCCL stream (shared) / on NCCL's default stream (shared-lowprio); auto = shared from 4 GPUs up, "
                         "where the host interface bounds the replicated upload (profiles/r2_e2e_upload_modes.txt)")
    ap.add_argument("--e2e-trace", action="store_true", help="add the per-batch event timeline of the host pipeline (rank 0) to the e2e object")
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl"],
                    help="N > 1: all-gather of the summaries fused into the filter kernel (NVLink peer stores) or NCCL after it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy (a fixed sample of "
                         f"at most {DUMP_MEMBERS} members), so that two builds can be compared output for output on identical inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def job_shape(a, world, rank):
    """(n_total, first member of this rank, members of this rank, scaling)"""
    from optistate_b200.distributed import shard_range

    if a.traj_total > 0:
        b, e = shard_range(a.traj_total, world, rank)
        return a.traj_total, b, e - b, "strong"
    return a.traj_per_gpu * world, rank * a.traj_per_gpu, a.traj_per_gpu, "weak"


def workload_config(a, world):
    n_total = a.traj_total if a.traj_total > 0 else a.traj_per_gpu * world
    per = f"{n_total} trajectories in the job ({n_total // world} per GPU)" if a.traj_total > 0 else f"{a.traj_per_gpu} trajectories per GPU"
    which = "BASELINE configs[3] as written" if n_total == 1 << 24 else "BASELINE configs[2]/[3] shape"
    return {
        "workload": f"monte-carlo noise sweep: {per} x {a.T} steps, {a.streams} shared base streams, per-member diagonal Q/R, "
                    f"summary outputs ({which}, {a.dtype})",
        "trajectories_per_gpu": n_total // world, "trajectories_total": n_total, "steps_per_trajectory": a.T,
        "base_streams": a.streams, "sharding": f"contiguous blocks x{world}, all-gather of summaries" if world > 1 else "single GPU",
        "covariance_structure": "decoupled groups (30 of 78 packed entries; exact zeros skipped)" if a.structure == "auto" else "full packed (78 entries)",
        "l2": "no explicit flush: per-iteration inputs (streams + per-member noise) exceed the 126 MB L2",
    }


Q_DIAG = np.array([0.01, 0.01, 0.01, 0.01, 0.0001, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.0001])  # settings.py:28
R_DIAG = np.full(10, 0.01)  # settings.py:30
BLOCK = 1 << 16


def mc_noise(first_member: int, count: int, n_streams: int):
    """Vectorised Monte-Carlo noise (same law as synth.monte_carlo_noise: 10**U(-0.5,0.5) per diagonal entry; the first
    pass over the streams stays nominal).  Drawn in blocks of 65,536 members so it is a function of the member id."""
    q = np.empty((12, count))
    r = np.empty((10, count))
    done = 0
    while done < count:
        m = first_member + done
        blk, off = divmod(m, BLOCK)
        n = min(BLOCK - off, count - done)
        rng = np.random.default_rng([10**6, blk])
        u = rng.uniform(-0.5, 0.5, (BLOCK, 22))[off:off + n]
        q[:, done:done + n] = (Q_DIAG[None, :] * 10.0 ** u[:, :12]).T
        r[:, done:done + n] = (R_DIAG[None, :] * 10.0 ** u[:, 12:]).T
        done += n
    ids = first_member + np.arange(count)
    nominal = ids < n_streams
    q[:, nominal] = Q_DIAG[:, None]
    r[:, nominal] = R_DIAG[:, None]
    return q, r


def parity_sample(st, q, r, stream_idx, summary_cols, nominal_x_steps=None):
    """Summary columns of a few members of a batch against the C oracle (oracle/kf_oracle.c) run on the same streams and
    noise.  st: base streams [T, C, S] (NumPy); q [12, n], r [10, n], stream_idx [n]; summary_cols [52, n] as the kernel
    wrote them.  Errors are max |difference| / max |oracle| per summary row, then the maximum over the rows of a group."""
    from oracle import c_oracle

    n = len(stream_idx)
    ref = c_oracle.run(st, n, Q=np.ascontiguousarray(q), R=np.ascontiguousarray(r), stream_index=np.asarray(stream_idx, np.int32),
                       noise_per_traj=True, want=("x_steps", "P_final", "nis_steps", "p_trace_steps", "k_gain_steps"))
    x = ref["x_steps"]  # [T, 12, n]
    T = x.shape[0]
    rows = {"x": (slice(0, 12), x[-1]), "p": (slice(12, 24), ref["P_final"][::13]),
            "nis": (slice(48, 49), ref["nis_steps"].mean(axis=0)[None]), "trace": (slice(49, 50), ref["p_trace_steps"][-1][None]),
            "gain": (slice(50, 51), ref["k_gain_steps"][-1][None]), "maxnis": (slice(51, 52), np.sqrt(ref["nis_steps"].max(axis=0))[None])}
    if "truth" in st:
        truth = st["truth"][:, :, stream_idx]
        rows["rmse"] = (slice(24, 36), np.sqrt(((x - truth) ** 2).mean(axis=0)))
    if nominal_x_steps is not None:
        nom = np.asarray(nominal_x_steps, np.float64)[:, :, stream_idx]
        rows["dev"] = (slice(36, 48), np.sqrt(((x - nom) ** 2).mean(axis=0)))
    got = np.asarray(summary_cols, np.float64)
    out = {"n": int(n), "steps": int(T)}
    for k, (sl, want) in rows.items():
        scale = np.abs(want).max(axis=1, keepdims=True)
        scale[scale == 0] = 1.0
        out["max_rel_" + k] = float((np.abs(got[sl] - want) / scale).max())
    return out


class ClockSampler:
    """SM clock / throttle reasons while the timed region runs (B200_PROFILING.md clocks line).

    One SYNCHRONOUS reading when the region is entered and one when it is left, so a region shorter than any polling
    period still has two samples (round 1 lost its only row that way), plus a polling thread every `period` seconds for
    long regions.  NVML (nvidia-ml-py, no subprocess) addressed by the PCI bus id of the CUDA device; if NVML is not
    usable the same readings come from one-shot `nvidia-smi --query-gpu` calls."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index: int, period: float = 0.1, bus_id: str | None = None):
        self.index, self.period, self.bus_id = index, period, bus_id
        self.sm, self.mx, self.reasons, self.how = [], [], set(), None
        self._nvml = self._handle = self._thread = None
        self._stop = threading.Event()
        self._lock = threading.Lock()

    # -- one reading -------------------------------------------------------------------------------------------
    def _open_nvml(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            if self.bus_id:
                try:
                    self._handle = pynvml.nvmlDeviceGetHandleByPciBusId(self.bus_id.encode())
                except Exception:
                    self._handle = None
            if self._handle is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                ids = [v for v in vis.split(",") if v.strip().isdigit()]
                phys = int(ids[self.index]) if self.index < len(ids) else self.index
                self._handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
            self.how = "nvml"
        except Exception:
            self._nvml = self._handle = None
            self.how = "nvidia-smi"

    def _read_nvml(self):
        n, h = self._nvml, self._handle
        sm = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
        mx = float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM))
        try:
            bits = int(n.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            bits = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        masks = (n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown,
                 n.nvmlClocksEventReasonSwThermalSlowdown, n.nvmlClocksEventReasonSwPowerCap)
        return sm, mx, [name for name, m in zip(self.NAMES, masks) if bits & m]

    def _read_smi(self):
        sel = self.bus_id if self.bus_id else str(self.index)
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", sel],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
        c = [v.strip() for v in out.split(",")]
        return float(c[0]), float(c[1]), [name for name, v in zip(self.NAMES, c[2:6]) if v.lower().startswith("active")]

    def sample(self):
        try:
            sm, mx, why = self._read_nvml() if self._nvml is not None else self._read_smi()
        except Exception:
            return
        with self._lock:
            self.sm.append(sm)
            self.mx.append(mx)
            self.reasons.update(why)

    # -- region --------------------------------------------------------------------------------------------------
    def _poll(self):
        while not self._stop.wait(self.period if self._nvml is not None else max(self.period, 1.0)):
            self.sample()

    def __enter__(self):
        self._open_nvml()
        self.sample()
        self._thread = threading.Thread(target=self._poll, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self.sample()  # the GPU has just finished the last timed step: clocks are still the ones it ran at
        self._stop.set()
        self._thread.join(timeout=25)

    def summary(self):
        with self._lock:
            sm, mx = list(self.sm), list(self.mx)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(self.reasons), "samples": len(sm), "how": self.how}


def cpu_port_rate(a, seconds_target=12.0, n_threads=0):
    """The oracle's C port of the reference filter (oracle/kf_oracle.c) on a bounded sample of the same workload:
    n_sample trajectories x T steps over the same base streams with Monte-Carlo noise.  Returns (steps/s, dict)."""
    from oracle import c_oracle
    from optistate_b200.synth import make_streams

    threads = n_threads or c_oracle.max_threads()
    S = min(a.streams, 64)
    st = make_streams(range(S), a.T)
    q, r = mc_noise(0, threads, S)
    t0 = time.perf_counter()
    c_oracle.run(st, threads, Q=q, R=r, n_threads=threads, want=("x_final",))  # calibration: one trajectory per thread
    dt = time.perf_counter() - t0
    per_thread = max(1, int(seconds_target / max(dt, 1e-3)))
    n = threads * min(per_thread, 64)
    q, r = mc_noise(0, n, S)
    t0 = time.perf_counter()
    c_oracle.run(st, n, Q=q, R=r, n_threads=threads, want=("x_final",))
    dt = time.perf_counter() - t0
    return n * a.T / dt, {"cores": threads, "kind": "port", "sample": f"{n} trajectories x {a.T} steps ({dt:.1f} s), C port of the reference filter "
                          f"(oracle/kf_oracle.c, pthreads, one block of trajectories per thread)"}


def reference_class_rates():
    """The unmodified reference class (oracle/_ref on the GPU box) on this box's host cores; {} when it is not staged."""
    try:
        from oracle import ref_timing

        return ref_timing.time_reference_class() or {"reference_class": "not staged (oracle/_ref missing)"}
    except Exception as e:  # noqa: BLE001
        return {"reference_class_error": str(e)[:200]}


def run_reference(a):
    """CPU arm: oracle C port with all host threads; a step = a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import c_oracle
    from optistate_b200.synth import make_streams

    threads = c_oracle.max_threads()
    S = min(a.streams, 64)
    st = make_streams(range(S), a.T)
    n = threads * 16
    q, r = mc_noise(0, n, S)
    last = {}
    fn = lambda: last.update(c_oracle.run(st, n, Q=q, R=r, n_threads=threads, want=("x_final",)))  # noqa: E731
    t0 = time.perf_counter()
    fn()
    first = time.perf_counter() - t0
    if first * (a.steps + a.warmup) > 240:  # keep the whole arm within a few minutes
        n = max(threads, int(n * 240 / (first * (a.steps + a.warmup))))
        q, r = mc_noise(0, n, S)
    for _ in range(max(a.warmup - 1, 0)):
        fn()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        fn()
    dt = time.perf_counter() - t0
    if a.dump_outputs:
        m = dump_members(n)
        dump_outputs(a.dump_outputs, {"x_final": last["x_final"][:, m], "members": m.astype(np.float64)})
    value = n * a.T * a.steps / dt
    sample = f"{n} trajectories x {a.T} steps per step over {S} base streams, Monte-Carlo Q/R"
    cpu = {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
    cpu.update(reference_class_rates())
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "strong" if a.traj_total > 0 else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(a, a.gpus), "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_native(a):
    import torch
    import torch.distributed as dist

    from optistate_b200 import fma_peak, kf_batch
    from optistate_b200 import _native as nv
    from optistate_b200.distributed import gather_columns, shard_range
    from optistate_b200.synth import make_streams

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float64 if a.dtype == "f64" else torch.float32
    esz = 8 if a.dtype == "f64" else 4
    T, S = a.T, a.streams
    n_total, first, n_local, scaling = job_shape(a, world, rank)

    # ---- synthetic inputs (host, pinned) -------------------------------------------------------------------
    st = make_streams(range(S), T)
    host = {k: torch.from_numpy(st[k]).to(dtype).pin_memory() for k in ("imu", "p", "dp", "contact", "f", "truth")}
    q_np, r_np = mc_noise(first, n_local, S)
    host["Q"] = torch.from_numpy(q_np).to(dtype).pin_memory()
    host["R"] = torch.from_numpy(r_np).to(dtype).pin_memory()
    del q_np, r_np
    d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
    # label stream 2: the nominal member of every stream (u = v = 0), one small launch, untimed
    nominal = kf_batch(d["imu"], d["p"], d["dp"], d["contact"], d["f"], dtype=dtype, outputs=("x_steps",), structure=a.structure).x_steps
    host["nominal"] = nominal.cpu().pin_memory()
    d["nominal"] = nominal
    out = {"summary": torch.empty((nv.SUMMARY_ROWS, n_local), dtype=dtype, device=dev),
           "status": torch.zeros(n_local, dtype=torch.int32, device=dev),
           "workspace": torch.empty(T * 10 * S * esz + 4 * S + 4096, dtype=torch.uint8, device=dev)}

    # N > 1: every GPU ends each step holding the summaries of ALL trajectories.  Default: the filter kernel stores them
    # into every GPU's copy itself (peer.PeerSummary); --gather nccl (or no peer access on this box): NCCL all-gather
    peer, gather_how = None, "single GPU"
    if world > 1:
        gather_how = "NCCL all-gather after the kernel"
        if a.gather == "fused":
            from optistate_b200.peer import PeerSummary
            try:
                peer = PeerSummary(n_total, dtype)
                gather_how = "fused into the filter kernel (NVLink peer stores) + one 4-byte NCCL all-reduce as barrier"
            except RuntimeError as e:  # agreed on by all ranks inside PeerSummary
                gather_how += f" ({e})"
    common = dict(Q=d["Q"], R=d["R"], n_traj=n_local, dtype=dtype, stream_offset=first, truth=d["truth"], nominal=d["nominal"],
                  outputs=("summary",), out=out, q_kind=nv.MAT_DIAG_PER, r_kind=nv.MAT_DIAG_PER, structure=a.structure)

    def step_nccl():
        res = kf_batch(d["imu"], d["p"], d["dp"], d["contact"], d["f"], **common)
        if world > 1:
            return gather_columns(res.summary, n_total)
        return res.summary

    def step_fused():
        peer.wait()  # every rank is done with the previous step's gathered array
        kf_batch(d["imu"], d["p"], d["dp"], d["contact"], d["f"], summary_peers=peer, **common)
        peer.wait()  # all kernels have finished: peer.tensor holds all n_total columns on every GPU
        return peer.tensor

    step_resident = step_fused if peer is not None else step_nccl

    # end-to-end through the public host-buffer API: every step uploads ALL of its inputs from pinned host memory and
    # downloads its summaries; the double-buffered pipeline overlaps step k+1's upload and step k-1's download with step
    # k's kernel, and the host reads each step's result one step later
    pipe = None
    e2e_state = {"prev": None, "sink": 0.0}

    def step_e2e():
        ticket = pipe.submit(host)
        if e2e_state["prev"] is not None:
            e2e_state["sink"] += float(pipe.result(e2e_state["prev"])[48, 0])  # the previous step's result, read on the host
        e2e_state["prev"] = ticket

    def finish_e2e():
        pipe.drain()
        e2e_state["sink"] += float(pipe.result(e2e_state["prev"])[48, 0])
        e2e_state["prev"] = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = nv.ext().launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()  # work queued on other streams must be inside the timed region
            torch.cuda.synchronize()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), nv.ext().launch_count() - l0

    for _ in range(a.warmup):
        step_resident()
    with ClockSampler(local, bus_id=_pci_bus_id(torch, local)) as clk:
        ms, launches = timed(step_resident, a.steps)
    steps_total = n_total * T * a.steps
    value = steps_total / (ms * 1e-3)
    status_bad = int((out["status"] != 0).sum().item())
    gathered = (peer.tensor if peer is not None else step_nccl()) if world > 1 else out["summary"]
    if rank == 0 and a.dump_outputs:
        # the gathered summary columns of a sample of the whole job's members; status words are per rank, so only those of
        # rank 0's own members (ids 0 .. n_local - 1) among them
        m = dump_members(n_total)
        mine = m[m < n_local]
        dump_outputs(a.dump_outputs, {"summary": gathered[:, torch.from_numpy(m).to(dev)].cpu().numpy(), "members": m.astype(np.float64),
                                      "status": out["status"][torch.from_numpy(mine).to(dev)].cpu().numpy().astype(np.float64),
                                      "status_members": mine.astype(np.float64)})

    # ---- parity of what was just timed: members of the timed batch against the C oracle (rank 0, outside the timed region).
    # First / last member, a nominal member, both sides of every shard boundary, and a few in between.
    parity = None
    if rank == 0:
        pick = {0, 5, S - 1, S, S + 17, n_total // 3, n_total - S, n_total - 1}
        for rk in range(1, world):
            b = shard_range(n_total, world, rk)[0] if a.traj_total > 0 else rk * n_local
            pick.update({b - 1, b})
        pick = np.array(sorted(m for m in pick if 0 <= m < n_total))
        qs = np.concatenate([mc_noise(int(m), 1, S)[0] for m in pick], axis=1)
        rs = np.concatenate([mc_noise(int(m), 1, S)[1] for m in pick], axis=1)
        if a.dtype == "f32":  # the kernel saw the noise rounded to FP32
            qs, rs = qs.astype(np.float32).astype(np.float64), rs.astype(np.float32).astype(np.float64)
        cols = gathered[:, torch.from_numpy(pick).to(dev)].cpu().numpy()
        parity = parity_sample(st, qs, rs, (pick % S).astype(np.int32), cols, nominal.cpu().numpy())
        parity["members"] = [int(m) for m in pick]
        tol_x, tol_p = (FP64_TOL, FP64_TOL) if a.dtype == "f64" else (FP32_TOL_X, FP32_TOL_P)
        parity["tolerance"] = {"x": tol_x, "p": tol_p}
        parity["ok"] = bool(parity["max_rel_x"] < tol_x and parity["max_rel_p"] < tol_p and
                            (a.dtype == "f32" or (parity["max_rel_rmse"] < 1e-9 and parity["max_rel_dev"] < 1e-7)))

    gather_info = None
    if world > 1:
        gather_info = {"how": gather_how}
        if peer is not None:
            # the same job with the NCCL all-gather, and a check that the two gathered arrays are identical
            fused_copy = peer.tensor.clone()
            for _ in range(2):
                ref = step_nccl()
            gather_info["identical_to_nccl_gather"] = bool(torch.equal(fused_copy, ref))
            ms_n, _ = timed(step_nccl, a.steps)
            gather_info["nccl_gather_value"] = steps_total / (ms_n * 1e-3)
            gather_info["nccl_gather_ms_per_step"] = ms_n / a.steps
            gather_info["peer_store_bytes_per_gpu_per_step"] = nv.SUMMARY_ROWS * esz * n_local * (world - 1)
            del fused_copy, ref

    # ---- measured FMA peak (roofline denominator): after the timed region, GPU at its loaded clocks, best of 3 x ~35 ms
    peak_flops = max(fma_peak(dtype, 1 << 21)[0] for _ in range(3))

    secondary = None
    if rank == 0 and not a.no_secondary:
        secondary = secondary_figures(a, torch, d, dev, dtype, st)

    e2e = None
    if not a.no_e2e:
        from optistate_b200.pipeline import KfHostPipeline

        # N > 1: the ranks filter different members of the SAME base streams; with --e2e-upload shared each uploads 1/N of the stream
        # arrays and the slices are exchanged over NVLink (pipeline.py); per-member noise and summaries are per rank
        exchange_group = None
        if a.e2e_upload == "auto":
            a.e2e_upload = "shared" if world >= 4 else "replicated"
        if world > 1 and a.e2e_upload != "replicated":
            from optistate_b200.distributed import stream_exchange_group

            try:
                exchange_group = stream_exchange_group() if a.e2e_upload == "shared" else dist.group.WORLD
            except Exception as e:  # a build of torch without the NCCL options: every rank fails alike and uploads everything itself
                print(f"bench: no high-priority exchange group ({e}); replicated upload", file=sys.stderr)
                exchange_group, a.e2e_upload = None, "replicated"
        pipe = KfHostPipeline(n_local, T, S, dtype=dtype, labels=("truth", "nominal"), stream_offset=first, structure=a.structure,
                              shared_streams_group=exchange_group, trace=a.e2e_trace)
        for _ in range(max(2, a.warmup - 1)):
            step_e2e()
        finish_e2e()
        ms_e, _ = timed(step_e2e, a.steps, finish=finish_e2e)
        # outside the timed region: the summaries the host received are those of the device-resident path, bit for bit (also what
        # checks the stream slices exchanged between the ranks in the shared upload mode)
        last = pipe.submit(host)
        got = pipe.result(last).clone()
        kf_batch(d["imu"], d["p"], d["dp"], d["contact"], d["f"], **common)
        torch.cuda.synchronize()
        e2e_same = bool(torch.equal(got, out["summary"].cpu()))
        if not e2e_same:
            raise SystemExit("bench: the host pipeline's summaries differ from the device-resident path's")
        h2d = pipe.h2d_bytes_per_batch  # counted from the copies this rank issued: all inputs at N = 1, its share of the streams + its noise at N > 1
        assert world > 1 or h2d == sum(host[k].numel() * host[k].element_size() for k in ("imu", "p", "dp", "contact", "f", "truth", "nominal", "Q", "R"))
        if world > 1:
            tot = torch.tensor([float(h2d), float(nv.SUMMARY_ROWS * n_local * esz)], dtype=torch.float64, device=dev)
            dist.all_reduce(tot)
            h2d_total, d2h_total = int(tot[0].item()), int(tot[1].item())
        else:
            h2d_total, d2h_total = h2d, nv.SUMMARY_ROWS * n_local * esz
        e2e = {"value": steps_total / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_total,
               "ms_per_step": ms_e / a.steps, "identical_to_resident_path": e2e_same, "upload": a.e2e_upload if world > 1 else "all inputs",
               "api": "optistate_b200.pipeline.KfHostPipeline (kf_batch on pinned host buffers, double-buffered)" +
                      ("; base streams uploaded once per job (1/N per rank) and all-gathered over NVLink" if pipe.world > 1 else "")}

    if e2e is not None and a.e2e_trace:
        e2e["timeline_ms"] = pipe.timeline()
    if peer is not None:
        peer.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    clocks = clk.summary()
    per_gpu = value / world
    sm_max = clocks.get("sm_max_mhz") or 1965.0
    sm_run = clocks.get("sm_mhz") or sm_max
    lanes = 64 if a.dtype == "f64" else 128
    n_sm = torch.cuda.get_device_properties(local).multi_processor_count
    theoretical_tf = n_sm * lanes * 2 * sm_max * 1e6 / 1e12      # at the maximum SM clock
    theoretical_run_tf = n_sm * lanes * 2 * sm_run * 1e6 / 1e12  # at the clock sampled during the timed region
    measured_tf = peak_flops / 1e12
    # the denominator: the issue peak measured in this run, unless it reads low against the pipe's arithmetic limit at the
    # sampled clock (round 1: 91.5 % - a cold, short probe); then the arithmetic limit, which is the stricter choice
    peak_tf, peak_src = (measured_tf, "measured in this run (optistate_fma_peak, best of 3 after the timed region)") \
        if measured_tf >= 0.98 * theoretical_run_tf else (theoretical_run_tf, f"{n_sm} SMs x {lanes} FMA/clk x 2 x sampled SM clock")
    prof = kernel_profile(a.dtype, a.structure)
    algorithmic_tf = per_gpu * FLOPS_ALGORITHMIC / 1e12
    executed_tf = per_gpu * prof["flops_executed"] / 1e12 if prof else None
    traffic = None
    if prof and prof["traffic_bytes"] is not None:
        per_block = 128 * prof["lanes"]
        if (n_local, T, S) == DEFAULT_SHAPE and prof["grid"] == (n_local + per_block - 1) // per_block:
            traffic = prof["traffic_bytes"]
    ms_step = ms / a.steps
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": a.dtype,
        "data": "synthetic", "config": workload_config(a, world), "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "roofline": {
            "bound": "fma", "unit": "TFLOP/s", "peak": peak_tf, "peak_source": peak_src,
            "achieved": executed_tf if executed_tf is not None else algorithmic_tf,
            "frac": (executed_tf if executed_tf is not None else algorithmic_tf) / peak_tf,
            "frac_is": "executed flops / peak" if executed_tf is not None else "ALGORITHMIC flops / peak (no ncu capture of this instantiation in profiles/)",
            "executed_flops_per_step": prof["flops_executed"] if prof else None,
            "fp_instructions_per_thread_step": prof["fp_instructions_per_thread_step"] if prof else None,
            "profile": {k: prof[k] for k in ("kernel", "source", "metrics_source", "fp_pipe_active_pct") if k in prof} if prof else None,
            "algorithmic_flops_per_step": FLOPS_ALGORITHMIC, "achieved_algorithmic": algorithmic_tf, "frac_algorithmic": algorithmic_tf / peak_tf,
            "measured_fma_peak_tflops": measured_tf, "theoretical_peak_tflops": theoretical_tf,
            "theoretical_peak_at_sampled_clock_tflops": theoretical_run_tf,
            "traffic": traffic, "algorithmic_bytes": algorithmic_bytes(n_local, T, S, esz),
            "hbm_gbs_algorithmic": algorithmic_bytes(n_local, T, S, esz) / (ms_step * 1e-3) / 1e9, "hbm_peak_gbs": _hbm_peak(),
            "note": "per GPU, dominant kernel kf_seq_tma_kernel (> 99 % of a step; the other launch is the measurement pre-pass). FMA-bound "
                    "(CUDA cores): HBM traffic is < 1 % of the copy peak because Monte-Carlo members share base streams through L2",
        },
        "parity_sample": parity, "status_nonzero_trajectories": status_bad, "secondary": secondary,
    }
    if gather_info is not None:
        line["gather"] = gather_info
        line["config"]["sharding"] = f"contiguous blocks x{world}; summaries gathered on every GPU: {gather_how}"
    if world == 1 and not a.no_cpu_baseline:
        v, info = cpu_port_rate(a)
        line["cpu_baseline"] = dict({"value": v, "unit": UNIT}, **info)
        line["cpu_baseline"].update(reference_class_rates())
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        raise SystemExit(f"bench.py: the timed batch does not match the oracle: {parity}")


def secondary_figures(a, torch, d, dev, dtype, st):
    """Rank 0, one GPU, outside the timed region; reported next to the headline, never part of it."""
    from optistate_b200 import kf_batch
    from optistate_b200 import _native as nv

    def once(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = float("inf")
        for _ in range(reps):
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) * 1e-3)
        return best

    T, S = a.T, a.streams
    sec = {}
    f64 = {k: (d[k] if dtype == torch.float64 else d[k].double()) for k in ("imu", "p", "dp", "contact", "f")}
    # BASELINE configs[1]: 1,024 trajectories x 10,000 steps, FP64, per-step estimates - a latency case (32 warps in flight)
    reps = max(1, 10000 // T)  # the streams repeated in time: the data content does not matter for the rate
    st2 = {k: v[:, :, :1024].repeat(reps, 1, 1).contiguous() for k, v in f64.items()}
    t2 = once(lambda: kf_batch(st2["imu"], st2["p"], st2["dp"], st2["contact"], st2["f"], outputs=("x_steps", "p_trace", "k_gain")))
    sec["cfg2_1024x10k_f64_steps_per_s"] = st2["imu"].shape[2] * st2["imu"].shape[0] / t2
    sec["cfg2_seconds"] = t2
    del st2
    # the general JOINT path (reference operand order, four lanes per trajectory) on 131,072 trajectories x 200 steps
    tj = once(lambda: kf_batch(f64["imu"][:200], f64["p"][:200], f64["dp"][:200], f64["contact"][:200], f64["f"][:200], n_traj=1 << 17,
                               algo="joint", outputs=("x_final",)))
    sec["joint_path_f64_steps_per_s"] = (1 << 17) * 200 / tj
    # the same sweep on all 78 packed covariance entries (the round-1 kernel), 262,144 trajectories x 300 steps, no summary
    for name, kw in (("sequential_full_cov_f64_steps_per_s", dict(structure="full")), ("sequential_decoupled_f64_steps_per_s", dict())):
        tf_ = once(lambda: kf_batch(f64["imu"][:300], f64["p"][:300], f64["dp"][:300], f64["contact"][:300], f64["f"][:300], n_traj=1 << 18,
                                    outputs=("x_final",), **kw))
        sec[name] = (1 << 18) * 300 / tf_
    if dtype == torch.float64 and S % 64 == 0:
        # BASELINE configs[2] verbatim: the FP32 sweep (packed two-trajectories-per-thread kernel), 1,048,576 x 1,000 with summaries
        n32 = 1 << 20
        q32, r32 = mc_noise(0, n32, S)
        f32 = {k: d[k].float() for k in ("imu", "p", "dp", "contact", "f", "truth", "nominal")}
        q32, r32 = torch.from_numpy(q32).to(dev, torch.float32), torch.from_numpy(r32).to(dev, torch.float32)
        t32 = once(lambda: kf_batch(f32["imu"], f32["p"], f32["dp"], f32["contact"], f32["f"], Q=q32, R=r32, n_traj=n32, dtype=torch.float32,
                                    truth=f32["truth"], nominal=f32["nominal"], outputs=("summary",), q_kind=nv.MAT_DIAG_PER, r_kind=nv.MAT_DIAG_PER), reps=2)
        sec["cfg3_fp32_1Mx1k_steps_per_s"] = n32 * T / t32
        sec["cfg3_fp32_seconds"] = t32
        del f32, q32, r32
    try:
        from optistate_b200.mpc import estimate_state_mpc_batch, mpc_forces
        from optistate_b200.synth import make_mpc_problems

        qp = [torch.from_numpy(v).to(dev) for v in make_mpc_problems(1 << 15)]
        tq = once(lambda: mpc_forces(*qp))
        trot = torch.where((torch.arange(1 << 15, device=dev) % 2 == 0)[None, :], torch.tensor([1.0, 0, 0, 1], device=dev, dtype=torch.float64)[:, None],
                           torch.tensor([0, 1.0, 1, 0], device=dev, dtype=torch.float64)[:, None]).contiguous()
        tqt = once(lambda: mpc_forces(qp[0], qp[1], qp[2], trot))
        stand = torch.ones((4, 1 << 15), dtype=torch.float64, device=dev)
        tqs = once(lambda: mpc_forces(qp[0], qp[1], qp[2], stand))
        sec["force_mpc_qps_per_s"] = (1 << 15) / tq
        sec["force_mpc_trot_qps_per_s"] = (1 << 15) / tqt
        sec["force_mpc_standing_qps_per_s"] = (1 << 15) / tqs
        # the closed loop the shipped driver runs (estimate_state_mpc: QP -> predict_mpc -> update, per step), 65,536 trajectories
        nc, tc = 1 << 16, 20
        rep = nc // min(S, nc)
        cl = {k: f64[k][:tc, :, :min(S, nc)].repeat(1, 1, rep).contiguous() for k in ("imu", "p", "dp", "contact")}
        body_ref = torch.zeros((tc, 5, 12, nc), dtype=torch.float64, device=dev)
        body_ref[:, :, 5] = 0.28
        fn = lambda: estimate_state_mpc_batch(cl["imu"], cl["p"], cl["dp"], cl["contact"], body_ref)  # noqa: E731
        tcl = once(fn, reps=2)
        sec["closed_loop_mpc_steps_per_s"] = nc * tc / tcl
        del cl, body_ref
    except Exception as e:  # noqa: BLE001 - a secondary figure must never take the headline down
        sec["force_mpc_error"] = str(e)[:300]
    try:
        sec.update(dropin_rate(st))
    except Exception as e:  # noqa: BLE001
        sec["dropin_error"] = str(e)[:300]
    return sec


def dropin_rate(st, steps=300, transfer=None):
    """The drop-in Kalman_Filter class stepped the way the reference driver steps it (one trajectory, host arrays in and out)."""
    from optistate_b200 import Kalman_Filter

    kf = Kalman_Filter()
    if transfer is not None:
        kf.transfer = transfer
    kf.x = kf.x.copy()
    cols = {k: [st[k][t, :, 0].reshape(-1, 1).copy() for t in range(steps)] for k in ("imu", "p", "dp", "contact", "f")}

    def run():
        for t in range(steps):
            imu = cols["imu"][t]
            kf.set_measurements(imu, kf.get_odom(cols["p"][t], cols["dp"][t], cols["contact"][t], imu))
            kf.predict(cols["p"][t].copy(), cols["f"][t])
            kf.update()
    run()
    best = float("inf")
    for _ in range(3):
        t0 = time.perf_counter()
        run()
        best = min(best, time.perf_counter() - t0)
    return {"dropin_class_steps_per_s": steps / best, "dropin_class_transfer": kf.transfer}


def _pci_bus_id(torch, local):
    """PCI address of CUDA device `local` in nvidia-smi / NVML notation (CUDA_VISIBLE_DEVICES may renumber devices)."""
    try:
        pr = torch.cuda.get_device_properties(local)
        return f"{pr.pci_domain_id:08X}:{pr.pci_bus_id:02X}:{pr.pci_device_id:02X}.0"
    except Exception:
        return None


def _hbm_peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        return 6650.0  # B200_PROFILING.md fallback


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)
