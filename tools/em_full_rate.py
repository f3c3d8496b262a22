"""Rates of the E-step on the full covariance (kf_noise_stats_full) on one GPU, in trajectory-steps/s, against the plain
full-covariance backward kernel.

    python tools/em_full_rate.py [--out profiles/r6_em_full_rate.txt] [--reps 3] [--only cfg1|mc]

Shapes and set-ups as in tools/smooth_full_rate.py: BASELINE configs[1] (1,024 x 10,000) and 65,536 x 1,000 over 1,024 streams,
predict() with a coupled P0 and predict_mpc with body_ref = the truth streams, FP64 and FP32.
  * end to end: CUDA events around whole kf_noise_stats_full calls (forward pass with full storage, z pre-pass, stats backward),
    after a warm-up call, with no smoothed outputs (what kf_noise_em_full runs each iteration);
  * a separate torch.profiler pass over kf_noise_stats_full and kf_smooth_full calls: kernel time of kf_rts_full_kernel<Real, mpc,
    true> (stats) against kf_rts_full_kernel<Real, mpc, false> (plain smoother, x_smooth + var_smooth);
  * the operation count of the added E-step work (em_full_flops, FMA = 2, as executed by all four warps) next to the plain step's
    (smooth_full_rate.rts_full_flops), over the FMA issue peak measured in the same run.
The card's name, power limit and SM clock are read in the same call.
"""
from __future__ import annotations

import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from smooth_full_rate import WARPS, cov_predict_full_flops, cov_predict_mpc_flops, ldl_flops, rts_full_flops, workload  # noqa: E402
from smooth_rate import RCP, ROT_PRODUCTS, SINCOS, card, copy_bandwidth  # noqa: E402


def em_full_flops(dt="f64", model="predict"):
    """Operations the E-step adds to one backward trajectory-step of kf_rts_full_kernel<Real, mpc, true>."""
    m_cols = 3 * (66 * 2 + 12 + 66 * 2)                   # per warp: three columns of (P-)^-1 by substitution on the factor
    quad = 3 * (12 * (1 + 11 * 2) + 12 * 2)               # per warp: m^T dPs m beside W = dPs G^T
    md = 3 * 12 * 3 + 3 * 6                               # per warp: (M d)_u with d re-formed, and the Sw accumulator
    sv = 10 * 5                                           # Sv: innovation of the smoothed state, square, variance, sum
    prior = 3 * SINCOS[dt] + ROT_PRODUCTS + 9 + (cov_predict_mpc_flops() + 9 if model == "mpc" else cov_predict_full_flops())
    ll = prior + ldl_flops(dt, 10) + 10 + 10 + 45 * 2 + 10 * 3 + 10 * 2 + 2  # one warp: P- again, L D L^T of S, solve, det
    return WARPS * (m_cols + quad + md) + sv + ll


def kernel_times(prof, reps):
    stats = plain = other = 0.0
    for ev in prof.key_averages():
        t = (ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total) * 1e-6
        if "kf_rts_full_kernel" in ev.key:
            args = ev.key.split("kf_rts_full_kernel<", 1)[1].split(">", 1)[0]
            if args.replace(" ", "").endswith(",true"):
                stats += t
            else:
                plain += t
        elif "kf_" in ev.key:
            other += t
    return stats / reps, plain / reps, other / reps


def measure(name, model, dtype, reps, peak, log):
    from torch.profiler import ProfilerActivity, profile

    from optistate_b200 import kf_noise_stats_full, kf_smooth_full

    dt = "f64" if dtype == torch.float64 else "f32"
    N, T, st, kw = workload(name, model, dtype)
    args = (st["imu"], st["p"], st["dp"], st["contact"], st["f"])
    out = {}
    run = lambda: kf_noise_stats_full(*args, dtype=dtype, out=out, **kw)  # noqa: E731
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
    smooth = lambda: kf_smooth_full(*args, dtype=dtype, outputs=("x_smooth", "var_smooth"), out=out, **kw)  # noqa: E731
    smooth()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            smooth()
        torch.cuda.synchronize()
    _, t_plain, _ = kernel_times(prof, reps)
    del out, st
    torch.cuda.empty_cache()
    steps = N * T
    nf = rts_full_flops(dt, model) + em_full_flops(dt, model)
    log(f"{name} {model} {dt}: N={N} T={T} storage {st_gb:.1f} GB")
    log(f"  kf_noise_stats_full end to end {total * 1e3:9.2f} ms/call  {steps / total:.3e} trajectory-steps/s")
    log(f"  forward + z pre-pass           {t_fwd * 1e3:9.2f} ms       {steps / t_fwd:.3e} trajectory-steps/s")
    log(f"  stats backward                 {t_stats * 1e3:9.2f} ms       {steps / t_stats:.3e} trajectory-steps/s "
        f"(kf_rts_full_kernel<{dt}, {model}, true>)")
    log(f"  plain backward                 {t_plain * 1e3:9.2f} ms       {steps / t_plain:.3e} trajectory-steps/s "
        f"(x_smooth + var_smooth); stats / plain = {t_stats / t_plain:.2f}")
    log(f"  stats ops {nf}/step executed (plain {rts_full_flops(dt, model)} + E-step {em_full_flops(dt, model)}, "
        f"x{nf / rts_full_flops(dt, model):.2f}) -> {nf * steps / peak[dt] * 1e3:.2f} ms at {peak[dt] / 1e12:.1f} TFLOP/s; "
        f"kernel reaches {nf * steps / peak[dt] / t_stats:.1%} of it")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default=None, help="cfg1 | mc (default: both)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("em_full_rate.py measures on a CUDA device; none found")
    from optistate_b200 import fma_peak

    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power limit, SM clock, max SM clock): {card()}")
    for model in ("predict", "mpc"):
        log(f"E-step operations added per trajectory-step ({model}): FP64 {em_full_flops('f64', model)}, FP32 "
            f"{em_full_flops('f32', model)} (plain backward {rts_full_flops('f64', model)}, {rts_full_flops('f32', model)})")
    log(f"device-to-device copy bandwidth (torch, 8 GiB, read + write): {copy_bandwidth() / 1e12:.2f} TB/s")
    peak = {"f64": fma_peak(torch.float64)[0], "f32": fma_peak(torch.float32)[0]}
    log(f"measured FMA issue peak: FP64 {peak['f64'] / 1e12:.1f} TFLOP/s, FP32 {peak['f32'] / 1e12:.1f} TFLOP/s")
    for name in (["cfg1", "mc"] if a.only is None else [a.only]):
        for model in ("predict", "mpc"):
            for dtype in (torch.float64, torch.float32):
                measure(name, model, dtype, a.reps, peak, log)
    log(f"card after the runs: {card()}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
