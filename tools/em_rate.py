"""Rates of the EM E-step (kf_noise_stats) on one GPU, in trajectory-steps/s, with the stats backward kernel's bounds.

    python tools/em_rate.py [--out profiles/r4_em_rate.txt] [--reps 3]

Shapes as in tools/smooth_rate.py: BASELINE configs[1] (1,024 trajectories x 10,000 steps) and the Monte-Carlo sweep (131,072 x
1,000 over 1,024 streams, per-member Q / R), in FP64 and FP32.
  * end to end: CUDA events around whole kf_noise_stats calls (forward pass with storage, z pre-pass, stats backward), after a
    warm-up call, with no smoothed outputs (what kf_noise_em runs each iteration);
  * a separate torch.profiler pass over kf_noise_stats and kf_smooth calls: kernel time of kf_rts_kernel<Real, true> (stats) against
    kf_rts_kernel<Real, false> (plain smoother, x_smooth + var_smooth);
  * bounds of the stats kernel, counted below: bytes (64 scalars read per step: x+, P+, x-, z; nothing written per step) over the
    device-to-device copy bandwidth measured in the same run, and operations (the plain backward step plus the E-step terms, FMA = 2)
    over 37.2 TFLOP/s FP64.
The card's name, power limit and SM clock are read in the same call.
"""
from __future__ import annotations

import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from smooth_rate import FP64_PEAK, RCP, card, copy_bandwidth, rts_bytes, rts_flops, workload  # noqa: E402


def sw_flops(n):
    """Sw of one group (rts_group<G, true>): column u of (P-)^-1 by substitution, (M d)_u, m^T dPs m, the accumulator."""
    f = 0
    for u in range(n):
        f += sum((k - u - 1) * 2 for k in range(u + 1, n))                                  # L f = e_u
        for k in range(n):                                                                 # back substitution
            f += (0 if k == u else 1) + 2 * len(range(k + 2 if k < u else k + 1, n))
        f += 1 + (n - 1) * 2                                                               # (M d)_u
        f += sum(1 + 2 + (1 + (k - 1) * 2 + 2 if k > 0 else 0) for k in range(n))          # m^T dPs m
        f += 1 + 2 + 2 + 1                                                                 # q^2 (quad + md^2) + q into acc
    return f


def ll_flops(nm, dt):
    """log N(y; 0, S) of one group: L D L^T of S solved on y, the quadratic form and the determinant product."""
    f = 2
    for j in range(nm):
        f += j + 1 + j * 2 + RCP[dt] + (nm - 1 - j) * (j * 2 + 1) + j * 2 + 1 + 2 + 1
    return f


def em_flops(dt="f64"):
    sv = 10 * (1 + 2 + 1) + 10  # Sv accumulators and the innovation
    return rts_flops(dt) + sv + sw_flops(6) + 3 * sw_flops(2) + ll_flops(6, dt) + 2 * ll_flops(1, dt) + ll_flops(2, dt)


def em_bytes(esz):
    return (12 + 30 + 12 + 10) * esz


def kernel_times(prof, reps):
    stats = plain = other = 0.0
    for ev in prof.key_averages():
        t = (ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total) * 1e-6
        if "kf_rts_kernel" in ev.key and "true" in ev.key:
            stats += t
        elif "kf_rts_kernel" in ev.key:
            plain += t
        elif "kf_" in ev.key:
            other += t
    return stats / reps, plain / reps, other / reps


def measure(name, dtype, reps, bw, log):
    from torch.profiler import ProfilerActivity, profile

    from optistate_b200 import kf_noise_stats, kf_smooth

    dt = "f64" if dtype == torch.float64 else "f32"
    esz = 8 if dt == "f64" else 4
    N, T, st, kw = workload(name)
    st = {k: v.to(dtype) for k, v in st.items()}
    if "Q" in kw:
        kw["Q"], kw["R"] = kw["Q"].to(dtype), kw["R"].to(dtype)
    args = (st["imu"], st["p"], st["dp"], st["contact"], st["f"])
    out = {}
    run = lambda: kf_noise_stats(*args, dtype=dtype, out=out, **kw)  # noqa: E731
    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    total = e0.elapsed_time(e1) * 1e-3 / reps
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run()
        torch.cuda.synchronize()
    t_stats, _, t_fwd = kernel_times(prof, reps)
    st_gb = out["em_storage"].numel() / 1e9
    del out
    torch.cuda.empty_cache()
    out = {}
    smooth = lambda: kf_smooth(*args, dtype=dtype, outputs=("x_smooth", "var_smooth"), out=out, **kw)  # noqa: E731
    smooth()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            smooth()
        torch.cuda.synchronize()
    _, t_plain, _ = kernel_times(prof, reps)
    del out
    torch.cuda.empty_cache()
    steps = N * T
    t_bw, t_fl = em_bytes(esz) * steps / bw, em_flops(dt) * steps / FP64_PEAK
    binding = "bandwidth" if t_bw >= t_fl else "compute (FP64 rate)"
    log(f"{name} {dt}: N={N} T={T} storage {st_gb:.1f} GB")
    log(f"  kf_noise_stats end to end {total * 1e3:9.2f} ms/call  {steps / total:.3e} trajectory-steps/s")
    log(f"  forward + z pre-pass      {t_fwd * 1e3:9.2f} ms       {steps / t_fwd:.3e} trajectory-steps/s")
    log(f"  stats backward            {t_stats * 1e3:9.2f} ms       {steps / t_stats:.3e} trajectory-steps/s (kf_rts_kernel<{dt}, true>)")
    log(f"  plain backward            {t_plain * 1e3:9.2f} ms       {steps / t_plain:.3e} trajectory-steps/s "
        f"(kf_rts_kernel<{dt}, false>, x_smooth + var_smooth); stats / plain = {t_stats / t_plain:.2f}")
    log(f"  stats bounds: bytes {em_bytes(esz)} B/step -> {t_bw * 1e3:.2f} ms at {bw / 1e12:.2f} TB/s; ops {em_flops(dt)} /step "
        f"(plain {rts_flops(dt)}, {rts_bytes(esz)} B) -> {t_fl * 1e3:.2f} ms at 37.2 TFLOP/s; binding: {binding}; "
        f"kernel reaches {max(t_bw, t_fl) / t_stats:.1%} of it")
    del st
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default=None, help="cfg1 | mc (default: both)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("em_rate.py measures on a CUDA device; none found")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power limit, SM clock, max SM clock): {card()}")
    log(f"stats backward operations per trajectory-step: FP64 {em_flops('f64')}, FP32 {em_flops('f32')} "
        f"(plain backward {rts_flops('f64')}, {rts_flops('f32')})")
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
