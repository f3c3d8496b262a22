"""Rates of the filter's adjoint (kf_vjp) on one GPU, in trajectory-steps/s, with the adjoint kernel's bounds.

    python tools/adjoint_rate.py [--out profiles/r9_adjoint_rate.txt] [--reps 10] [--windows 5]

Shapes as in tools/smooth_rate.py: the Monte-Carlo sweep (131,072 x 1,000 over 1,024 streams, per-member Q / R) and BASELINE
configs[1] (1,024 trajectories x 10,000 steps), in FP64 and FP32; both work sets are far larger than the 126 MB L2.
  * end to end: CUDA events around whole kf_vjp calls (forward pass with storage, z and moment pre-pass, adjoint), after a warm-up,
    in `windows` timed windows of `reps` calls each: the median per-call time and the spread (min - max) over the windows;
  * the split: a separate torch.profiler pass over the same calls, kernel time of kf_adjoint_kernel against the forward kernels;
  * bounds of the adjoint kernel, counted below from its loops: bytes (74 scalars read per step: th+, P+, x- at the measured
    states, x_bar, z, C; nothing written per step) over the device-to-device copy bandwidth measured in the same run, and
    operations (FMA = 2) over the FMA peak of the same precision measured in the same run (optistate_fma_peak).
The card's name, power limit and SM clock are read in the same call.
"""
from __future__ import annotations

import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smooth_rate import RCP, ROT_PRODUCTS, SINCOS, card, copy_bandwidth, cov_predict_flops, workload  # noqa: E402


def adj_group_flops(n, m, dt):
    """adj_group<G> (kf_adjoint.cuh) on a group of n states with m measured; FMA = 2."""
    h = n // 2
    f = 0
    for j in range(m):                                                   # L D L^T of S
        f += j + 1 + j * 2 + RCP[dt] + (m - 1 - j) * (j * 2 + 1)
    for c in range(m):                                                   # S^-1, column c
        f += sum((k - c) * 2 for k in range(c, m)) + sum(1 + (m - 1 - k) * 2 for k in range(m))
    f += n * n if m == n else n * m * (1 + (m - 1) * 2) + n * m          # A (and K)
    f += m * (m + n) * 2 + n * n * 2                                     # v, b, A^T a
    f += m * (1 + n * (n * 2 + 2) + 1)                                   # rb
    f += sum(n * n * 2 + (n - j) * (n * 2 + 5) for j in range(n))       # Pb = A^T Pi A + sym(at w^T)
    f += n                                                               # qb
    if n == 6:                                                           # th-term and J^T for {th, w}
        f += 18 + 9 * 3 * 2 + 9 * 2 + 9 * (6 * 2 + 2 + 3 * 2)
    else:
        f += 2
    f += sum(n * (h * 2 if j >= h else 0) + sum(h * 2 for i in range(j, n) if i >= h) for j in range(n))  # Pi = F^T Pb F
    return f


def adj_flops(dt="f64"):
    """One reverse step: a += x_bar, y, R and its derivatives (a second sincos set), dw'/dth, P-, then the four groups."""
    jw = 3 * 6 * 2 + 3 + 3 * (3 * 6 * 2 + 3 + 3 * 3 * 4)
    f = 12 + 10 + 2 * 3 * SINCOS[dt] + ROT_PRODUCTS + 9 + jw + cov_predict_flops() + 9
    return f + adj_group_flops(6, 6, dt) + 2 * adj_group_flops(2, 1, dt) + adj_group_flops(2, 2, dt)


def adj_bytes(esz):
    return (3 + 30 + 10 + 12 + 10 + 9) * esz


def kernel_times(prof, reps):
    adj = other = 0.0
    for ev in prof.key_averages():
        t = (ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total) * 1e-6
        if "kf_adjoint_kernel" in ev.key:
            adj += t
        elif "kf_" in ev.key:
            other += t
    return adj / reps, other / reps


def measure(name, dtype, reps, windows, bw, peak, log):
    from torch.profiler import ProfilerActivity, profile

    from optistate_b200 import kf_vjp

    dt = "f64" if dtype == torch.float64 else "f32"
    esz = 8 if dt == "f64" else 4
    N, T, st, kw = workload(name)
    st = {k: v.to(dtype) for k, v in st.items()}
    if "Q" in kw:
        kw["Q"], kw["R"] = kw["Q"].to(dtype), kw["R"].to(dtype)
    args = (st["imu"], st["p"], st["dp"], st["contact"], st["f"])
    xbar = torch.randn((T, 12, N), dtype=dtype, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    out = {}
    run = lambda: kf_vjp(*args, dtype=dtype, grad_x_steps=xbar, out=out, **kw)  # noqa: E731
    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_call = []
    for _ in range(windows):
        e0.record()
        for _ in range(reps):
            run()
        e1.record()
        torch.cuda.synchronize()
        per_call.append(e0.elapsed_time(e1) * 1e-3 / reps)
    per_call.sort()
    total = per_call[len(per_call) // 2]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run()
        torch.cuda.synchronize()
    t_adj, t_fwd = kernel_times(prof, reps)
    st_gb = out["adj_storage"].numel() / 1e9
    del out, xbar
    torch.cuda.empty_cache()
    steps = N * T
    ops = adj_flops(dt)
    t_bw, t_fl = adj_bytes(esz) * steps / bw, ops * steps / peak
    binding = "bandwidth" if t_bw >= t_fl else "compute"
    log(f"{name} {dt}: N={N} T={T} storage {st_gb:.1f} GB")
    log(f"  kf_vjp end to end            {total * 1e3:9.2f} ms/call  {steps / total:.3e} trajectory-steps/s (median of {windows} "
        f"windows of {reps} calls; spread {per_call[0] * 1e3:.2f} - {per_call[-1] * 1e3:.2f} ms/call)")
    log(f"  forward with storage + pre-pass {t_fwd * 1e3:6.2f} ms       {steps / t_fwd:.3e} trajectory-steps/s")
    log(f"  adjoint                      {t_adj * 1e3:9.2f} ms       {steps / t_adj:.3e} trajectory-steps/s (kf_adjoint_kernel<{dt}>)")
    log(f"  adjoint bounds: bytes {adj_bytes(esz)} B/step -> {t_bw * 1e3:.2f} ms at {bw / 1e12:.2f} TB/s; ops {ops} /step -> "
        f"{t_fl * 1e3:.2f} ms at the measured {dt} FMA peak {peak / 1e12:.1f} TFLOP/s; binding: {binding}; kernel reaches "
        f"{max(t_bw, t_fl) / t_adj:.1%} of it")
    del st
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--only", default=None, help="mc | cfg1 (default: both)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("adjoint_rate.py measures on a CUDA device; none found")
    from optistate_b200 import fma_peak

    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power limit, SM clock, max SM clock): {card()}")
    log(f"adjoint operations per trajectory-step: FP64 {adj_flops('f64')}, FP32 {adj_flops('f32')}; "
        f"bytes read per trajectory-step: FP64 {adj_bytes(8)}, FP32 {adj_bytes(4)}")
    bw = copy_bandwidth()
    log(f"device-to-device copy bandwidth (torch, 8 GiB, read + write): {bw / 1e12:.2f} TB/s")
    peaks = {torch.float64: fma_peak(torch.float64, 1 << 18)[0], torch.float32: fma_peak(torch.float32, 1 << 20)[0]}
    log(f"measured FMA peak (optistate_fma_peak): FP64 {peaks[torch.float64] / 1e12:.1f} TFLOP/s, "
        f"FP32 {peaks[torch.float32] / 1e12:.1f} TFLOP/s")
    for name in (["mc", "cfg1"] if a.only is None else [a.only]):
        for dtype in (torch.float64, torch.float32):
            measure(name, dtype, a.reps, a.windows, bw, peaks[dtype], log)
    log(f"card after the runs: {card()}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
