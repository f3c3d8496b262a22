"""Rates of the full-covariance smoother (kf_smooth_full) on one GPU, in trajectory-steps/s, with the backward kernel's bounds.

    python tools/smooth_full_rate.py [--out profiles/r5_smooth_full_rate.txt] [--reps 3] [--only cfg1|mc]

Shapes: BASELINE configs[1] (1,024 trajectories x 10,000 steps, one stream each) and a Monte-Carlo shape that fits the storage
(65,536 x 1,000 over 1,024 streams: 41 GB of P+ in FP64), each in FP64 and FP32 and under both covariance models (predict() with a
coupled P0, predict_mpc with body_ref = the truth streams); every work set is far larger than the 126 MB L2.
  * end to end: CUDA events around whole kf_smooth_full calls (forward pass with full storage + backward kernel), after a warm-up;
  * the split: a separate torch.profiler pass over the same calls, kernel time of kf_rts_full_kernel against everything else;
  * bounds of the backward kernel, from code below: bytes moved per trajectory-step (x+, P+, x- and the reference angles read,
    x_smooth and var_smooth written) over the device-to-device copy bandwidth measured in the same run, and the operation count
    of the kernel's arithmetic (rts_full_flops, FMA = 2; as executed, i.e. with the four warps' redundant P- and L D L^T) over
    the FMA issue peak measured in the same run (optistate_fma_peak) for the dtype.
The card's name, power limit and SM clock are read in the same call.
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from smooth_rate import RCP, ROT_PRODUCTS, SINCOS, card, copy_bandwidth  # noqa: E402

WARPS = 4  # roles per trajectory in kf_rts_full_kernel; each recomputes P- and its factor


def cov_predict_full_flops():
    """cov_predict_sym<false>: A = dt R^T (9), 156 FMAs of the two factors, + diag(q) (12)."""
    return 9 + 156 * 2 + 12


def cov_predict_mpc_flops():
    """cov_predict_mpc_sym: row sums (132) and their sum (11), v (18), U (45), the 6x6 block of D P D^T (96), the 78 entries (132)."""
    return 132 + 11 + 18 + 45 + 96 + 132


def ldl_flops(dt, n=12):
    f = 0
    for j in range(n):
        f += j + j * 2 + RCP[dt] + (n - 1 - j) * (j * 2 + 1)
    return f


def rts_full_flops(dt="f64", model="predict", executed=True):
    """Operations of one backward trajectory-step of kf_rts_full_kernel.  The exponentials of the mpc transition count one each."""
    per_warp = 3 * SINCOS[dt] + ROT_PRODUCTS + 9 + ldl_flops(dt)  # rotation, B, L D L^T
    per_warp += cov_predict_mpc_flops() + 9 if model == "mpc" else cov_predict_full_flops()
    cols = 3 * (3 * 3 * 2 + 3 * 2 + (23 if model == "mpc" else 0))  # this warp's columns of C = F P+
    cols += 3 * (66 * 2 + 12 + 66 * 2)                                # their solves
    cols += 12 + 3 * 12 * 2                                           # d, xs
    cols += 12 * 3 * (1 + 11 * 2)                                     # W = dPs G^T
    shared = 78 + 78 * 12 * 2                                         # dPs, the Ps triangle
    return (WARPS if executed else 1) * per_warp + WARPS * cols + shared


def rts_full_bytes(esz, model):
    return (12 + 78 + 12 + (3 if model == "mpc" else 0) + 24) * esz


def workload(name, model, dtype):
    from oracle import cases
    from optistate_b200.synth import make_streams

    N, T, S = (1024, 10000, 1024) if name == "cfg1" else (65536, 1000, 1024)
    st = {k: torch.from_numpy(v).cuda().to(dtype) for k, v in make_streams(range(S), T).items()}
    if model == "mpc":
        kw = dict(cov_model="mpc", body_ref=st["truth"])
    else:
        rng = np.random.default_rng(77)
        A = rng.standard_normal((12, 12))
        kw = dict(P0=0.02 * (A @ A.T / 12 + 0.5 * np.eye(12)))
    kw.update(n_traj=N, Q=cases.Q_DEFAULT, R=cases.R_DEFAULT)
    return N, T, st, kw


def measure(name, model, dtype, reps, bw, peak, log):
    from optistate_b200 import kf_smooth_full

    dt = "f64" if dtype == torch.float64 else "f32"
    esz = 8 if dt == "f64" else 4
    N, T, st, kw = workload(name, model, dtype)
    args = (st["imu"], st["p"], st["dp"], st["contact"], st["f"])
    out = {}
    run = lambda: kf_smooth_full(*args, dtype=dtype, outputs=("x_smooth", "var_smooth"), out=out, **kw)  # noqa: E731
    run()  # warm-up: module load, storage and output allocation
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    total = e0.elapsed_time(e1) * 1e-3 / reps
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run()
        torch.cuda.synchronize()
    back = fwd = 0.0
    for ev in prof.key_averages():
        t = ev.device_time_total * 1e-6 if hasattr(ev, "device_time_total") else ev.cuda_time_total * 1e-6
        if "kf_rts_full_kernel" in ev.key:
            back += t
        elif "kf_" in ev.key:
            fwd += t
    back, fwd = back / reps, fwd / reps
    steps = N * T
    nb, nf = rts_full_bytes(esz, model), rts_full_flops(dt, model)
    t_bw, t_fl = nb * steps / bw, nf * steps / peak[dt]
    binding = "bandwidth" if t_bw >= t_fl else "compute"
    log(f"{name} {model} {dt}: N={N} T={T} storage {out['smooth_storage'].numel() / 1e9:.1f} GB")
    log(f"  end to end  {total * 1e3:9.2f} ms/call  {steps / total:.3e} trajectory-steps/s")
    log(f"  forward     {fwd * 1e3:9.2f} ms        {steps / fwd:.3e} trajectory-steps/s (full-covariance filter + P+ / x+ / x- stores)")
    log(f"  backward    {back * 1e3:9.2f} ms        {steps / back:.3e} trajectory-steps/s (kf_rts_full_kernel)")
    log(f"  backward bounds: bytes {nb} B/step -> {t_bw * 1e3:.2f} ms at {bw / 1e12:.2f} TB/s; ops {nf}/step executed "
        f"({rts_full_flops(dt, model, False)} without the redundant P- / factor) -> {t_fl * 1e3:.2f} ms at {peak[dt] / 1e12:.1f} TFLOP/s; "
        f"binding: {binding}; kernel reaches {max(t_bw, t_fl) / back:.1%} of it")
    del out, st
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default=None, help="cfg1 | mc (default: both)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("smooth_full_rate.py measures on a CUDA device; none found")
    from optistate_b200 import fma_peak

    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power limit, SM clock, max SM clock): {card()}")
    for model in ("predict", "mpc"):
        log(f"backward operations per trajectory-step ({model}): FP64 {rts_full_flops('f64', model)}, FP32 {rts_full_flops('f32', model)}")
    bw = copy_bandwidth()
    log(f"device-to-device copy bandwidth (torch, 8 GiB, read + write): {bw / 1e12:.2f} TB/s")
    peak = {"f64": fma_peak(torch.float64)[0], "f32": fma_peak(torch.float32)[0]}
    log(f"measured FMA issue peak: FP64 {peak['f64'] / 1e12:.1f} TFLOP/s, FP32 {peak['f32'] / 1e12:.1f} TFLOP/s")
    for name in (["cfg1", "mc"] if a.only is None else [a.only]):
        for model in ("predict", "mpc"):
            for dtype in (torch.float64, torch.float32):
                measure(name, model, dtype, a.reps, bw, peak, log)
    log(f"card after the runs: {card()}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
