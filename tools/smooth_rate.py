"""Rates of the fixed-interval smoother (kf_smooth) on one GPU, in trajectory-steps/s, with the backward kernel's bounds.

    python tools/smooth_rate.py [--out profiles/r3_smooth_rate.txt] [--reps 3]

Shapes: BASELINE configs[1] (1,024 trajectories x 10,000 steps, one stream each) and a Monte-Carlo sweep (131,072 x 1,000 over
1,024 streams, per-member Q / R), each in FP64 and FP32; both work sets are far larger than the 126 MB L2.
  * end to end: CUDA events around whole kf_smooth calls (forward pass with storage + backward kernel), after a warm-up call;
  * the split: a separate torch.profiler pass over the same calls, kernel time of kf_rts_kernel against everything else;
  * bounds of the backward kernel, from code below: bytes moved (54 scalars read per step, 24 written: x_smooth + var_smooth) over
    the device-to-device copy bandwidth measured in the same run with torch copies, and the exact operation count of the kernel's
    arithmetic (rts_flops, FMA = 2) over 37.2 TFLOP/s FP64 (the data sheet's FP64 rate; FP32 uses the same kernel shape, so its
    compute bound is reported against the same figure for comparison only).
The card's name, power limit and SM clock are read in the same call.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FP64_PEAK = 37.2e12

# ---- exact operation count of one backward step of kf_rts_kernel (kf_smooth.cuh); FMA = 2 flops, rint / compares not counted
SINCOS = {"f64": 1 + 4 * 2 + 1 + 5 * 2 + 1 + 2 + 5 * 2 + 1 + 1 + 2 + 1, "f32": 1 + 3 * 2 + 1 + 2 * 2 + 1 + 2 + 2 * 2 + 1 + 1 + 2 + 1}
RCP = {"f64": 3 * 2, "f32": 2 * 2}  # the FMAs that refine the hardware seed (rcp_, kf_arith.cuh)
ROT_PRODUCTS = 21  # rot_zyx: products and sums of the multiplied-out R


def cov_predict_flops():
    """cov_predict_sym<true>: A = dt R^T (9), the coupled FMAs of the two factors (72), + diag(q) (12)."""
    return 9 + 72 * 2 + 12


def group_flops(n, dt):
    h = n // 2
    f = h * n * h * 2                                              # C = F P+
    for j in range(n):                                             # LDL^T
        f += j + j * 2 + RCP[dt] + (n - 1 - j) * (j * 2 + 1)
    f += n * (n * (n - 1) // 2 * 2 + n + n * (n - 1) // 2 * 2)     # n forward / scale / back substitutions
    f += n * n * 2                                                 # xs = x+ + G d
    for j in range(n):                                             # G dPs G^T, lower triangle
        f += n * (1 + (n - 1) * 2) + (n - j) * n * 2
    return f


def rts_flops(dt="f64"):
    f = 3 * SINCOS[dt] + ROT_PRODUCTS + cov_predict_flops() + 9 + 30 + 12  # rotation, P-, A, dPs, d
    return f + group_flops(6, dt) + 3 * group_flops(2, dt)


def rts_bytes(esz, var=True):
    return (12 + 30 + 12 + 12 + (12 if var else 0)) * esz


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q.splitlines()[0] if q else torch.cuda.get_device_name()


def copy_bandwidth(nbytes=8 << 30, reps=10):
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3
    del a, b
    torch.cuda.empty_cache()
    return 2 * nbytes * reps / s  # read + write


def workload(name):
    from oracle import cases
    from optistate_b200.synth import make_streams, monte_carlo_noise

    if name == "cfg1":
        N, T, S = 1024, 10000, 1024
        st = make_streams(range(S), T)
        kw = dict(n_traj=N)
    else:
        N, T, S = 131072, 1000, 1024
        st = make_streams(range(S), T)
        q, r = monte_carlo_noise(np.arange(N), np.diag(cases.Q_DEFAULT), np.diag(cases.R_DEFAULT))
        kw = dict(n_traj=N, Q=torch.from_numpy(q).cuda(), R=torch.from_numpy(r).cuda())
    return N, T, {k: torch.from_numpy(v).cuda() for k, v in st.items()}, kw


def measure(name, dtype, reps, bw, log):
    from optistate_b200 import kf_smooth

    dt = "f64" if dtype == torch.float64 else "f32"
    esz = 8 if dt == "f64" else 4
    N, T, st, kw = workload(name)
    st = {k: v.to(dtype) for k, v in st.items()}
    if "Q" in kw:
        kw["Q"], kw["R"] = kw["Q"].to(dtype), kw["R"].to(dtype)
    args = (st["imu"], st["p"], st["dp"], st["contact"], st["f"])
    out = {}
    run = lambda: kf_smooth(*args, dtype=dtype, outputs=("x_smooth", "var_smooth"), out=out, **kw)  # noqa: E731
    run()  # warm-up: module load, storage and output allocation
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    total = e0.elapsed_time(e1) * 1e-3 / reps
    # kernel split in a separate, profiled pass
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run()
        torch.cuda.synchronize()
    back = fwd = 0.0
    for ev in prof.key_averages():
        t = ev.device_time_total * 1e-6 if hasattr(ev, "device_time_total") else ev.cuda_time_total * 1e-6
        if "kf_rts_kernel" in ev.key:
            back += t
        elif "kf_" in ev.key:
            fwd += t
    back, fwd = back / reps, fwd / reps
    steps = N * T
    b_bytes, b_flops = rts_bytes(esz) * steps, rts_flops(dt) * steps
    t_bw, t_fl = b_bytes / bw, b_flops / FP64_PEAK
    binding = "bandwidth" if t_bw >= t_fl else "compute (FP64 rate)"
    st_gb = out["smooth_storage"].numel() / 1e9
    log(f"{name} {dt}: N={N} T={T} storage {st_gb:.1f} GB")
    log(f"  end to end  {total * 1e3:9.2f} ms/call  {steps / total:.3e} trajectory-steps/s")
    log(f"  forward     {fwd * 1e3:9.2f} ms        {steps / fwd:.3e} trajectory-steps/s (filter + packed P+ / x+ / x- stores)")
    log(f"  backward    {back * 1e3:9.2f} ms        {steps / back:.3e} trajectory-steps/s (kf_rts_kernel)")
    log(f"  backward bounds: bytes {rts_bytes(esz)} B/step -> {t_bw * 1e3:.2f} ms at {bw / 1e12:.2f} TB/s; "
        f"ops {rts_flops(dt)} /step -> {t_fl * 1e3:.2f} ms at 37.2 TFLOP/s; binding: {binding}; "
        f"kernel reaches {max(t_bw, t_fl) / back:.1%} of it")
    del out, st
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default=None, help="cfg1 | mc (default: both)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("smooth_rate.py measures on a CUDA device; none found")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power limit, SM clock, max SM clock): {card()}")
    log(f"backward operation count per trajectory-step: FP64 {rts_flops('f64')}, FP32 {rts_flops('f32')}")
    bw = copy_bandwidth()
    log(f"device-to-device copy bandwidth (torch, 8 GiB, read + write): {bw / 1e12:.2f} TB/s")
    for name in (["cfg1", "mc"] if a.only is None else [a.only]):
        for dtype in (torch.float64, torch.float32):
            measure(name, dtype, a.reps, bw, log)
    log(f"card after the runs: {card()}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
