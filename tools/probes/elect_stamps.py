"""Developer probe: what the refill election of the streamed filter costs a warp, and how the warps of one scheduler sit in phase.

    python tools/probes/elect_stamps.py build DIR   (no GPU needed) liboptistate_kf.so into DIR, its FP64 decoupled-group kernels
                                                    (kf_seq_tma_f64_sum_blk.cu) compiled with -DOKF_ELECT_STAMPS
    python tools/probes/elect_stamps.py run DIR     (GPU) one bench.py-shaped launch through DIR's library, then the analysis

The bench shape: 1 M members x 1,000 steps, 1,024 shared streams, per-member Q and R, summary against truth and nominal, FP64,
so the launch runs kf_seq_tma_kernel<double, summary, 0, 0, decoupled groups>.  Lane 0 of each warp of the first 1,024 blocks stamps
clock64() at the top of steps 400-415, around each of the three refill elections (election and copy issue) and at the end of the
step (kf_seq_tma.cuh, OKF_STAMP).  clock64 counts SM cycles and is comparable between warps
of one SM only, so phases are compared between blocks that ran on the same SM.

Reported (cycles, from the stamps):
  step      stamp(kStTop, t + 1) - stamp(kStTop, t) per warp: the step time of one warp, from which the throughput kernel's rate
            per scheduler is  warps per scheduler x 1 / step
  elect g   stamp(kStElect{g}End) - stamp(kStElect{g}): what the election of group g, and the copy issue when this warp is the last
            reader, cost the warp (in a build with the stamps: they fence the span)
  phase     for the blocks that started on one SM together: (top_b(t) - top_a(t)) mod step / step of warp w of blocks a, b; 0 or
            1 = lockstep
"""
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
BLOCKS, WARPS, T0, STEPS, EVENTS = 1024, 4, 400, 16, 8  # kf_seq_tma.cuh, OKF_ELECT_STAMPS
EV = ["top", "elect0", "elect0_end", "elect1", "elect1_end", "elect2", "elect2_end", "end"]


def build(out: str) -> None:
    sys.path.insert(0, ROOT)
    from optistate_b200 import _build

    _build.build_kf_lib()
    os.makedirs(out, exist_ok=True)
    tu = "kf_seq_tma_f64_sum_blk"
    obj = os.path.join(out, tu + ".o")
    subprocess.check_call([_build._nvcc(), *_build.NVCC_FLAGS, "-DOKF_ELECT_STAMPS", "-c", "-o", obj, os.path.join(_build.CSRC, tu + ".cu")])
    others = [os.path.join(_build.OBJ_DIR, o) for o in sorted(os.listdir(_build.OBJ_DIR)) if o.endswith(".o") and o != tu + ".o"]
    subprocess.check_call([_build._nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o",
                           os.path.join(out, "liboptistate_kf.so"), *others, obj])
    os.remove(obj)
    print("built", os.path.join(out, "liboptistate_kf.so"))


def run(libdir: str) -> None:
    libdir = os.path.abspath(libdir)
    if os.environ.get("LD_LIBRARY_PATH", "").split(":")[0] != libdir:  # the extension must bind to this library: set before start-up
        os.environ["LD_LIBRARY_PATH"] = libdir + ":" + os.environ.get("LD_LIBRARY_PATH", "")
        os.execv(sys.executable, [sys.executable] + sys.argv)
    import torch

    sys.path.insert(0, ROOT)
    from optistate_b200 import _native as nv
    from optistate_b200 import kf_batch
    from optistate_b200.synth import make_streams

    lib = ctypes.CDLL(os.path.join(libdir, "liboptistate_kf.so"))
    if not hasattr(lib, "okf_elect_stamps_read"):
        raise SystemExit(f"{libdir}/liboptistate_kf.so was not built with -DOKF_ELECT_STAMPS")
    N, T, S = 1 << 20, 1000, 1024
    st = make_streams(range(S), T)
    rng = np.random.default_rng(0)
    dev = {k: torch.from_numpy(v).to("cuda", torch.float64) for k, v in st.items()}
    q = torch.from_numpy(0.01 * 10 ** rng.uniform(-0.5, 0.5, (12, N))).cuda()
    r = torch.from_numpy(0.01 * 10 ** rng.uniform(-0.5, 0.5, (10, N))).cuda()
    kw = dict(Q=q, R=r, q_kind=nv.MAT_DIAG_PER, r_kind=nv.MAT_DIAG_PER, n_traj=N, dtype=torch.float64, outputs=("summary",),
              truth=dev["truth"], nominal=dev["truth"] * 0.5)
    for _ in range(2):  # the second launch is the one read back
        kf_batch(dev["imu"], dev["p"], dev["dp"], dev["contact"], dev["f"], **kw)
    torch.cuda.synchronize()
    stamps = np.zeros(BLOCKS * WARPS * STEPS * EVENTS, np.int64)
    smid = np.zeros(BLOCKS, np.uint32)
    assert lib.okf_elect_stamps_read(stamps.ctypes.data_as(ctypes.c_void_p), smid.ctypes.data_as(ctypes.c_void_p)) == 0
    analyse(stamps.reshape(BLOCKS, WARPS, STEPS, EVENTS), smid, torch.cuda.get_device_name())


def analyse(s: np.ndarray, smid: np.ndarray, device: str) -> None:
    ok = (s[:, :, :, 0] > 0).all(axis=(1, 2))
    s, smid = s[ok], smid[ok]
    print(f"device: {device}; {len(s)} blocks stamped, steps {T0}-{T0 + STEPS - 1}, 4 warps each")
    step = np.diff(s[:, :, :, 0], axis=2)
    print(f"step (cycles per warp-step): median {np.median(step):.0f}, p10 {np.percentile(step, 10):.0f}, p90 {np.percentile(step, 90):.0f}")

    def span(a, b):
        d = s[:, :, :, EV.index(b)] - s[:, :, :, EV.index(a)]
        d = d[(s[:, :, :, EV.index(a)] > 0) & (s[:, :, :, EV.index(b)] > 0)]
        return d

    total = 0.0
    for a, b in (("elect0", "elect0_end"), ("elect1", "elect1_end"), ("elect2", "elect2_end")):
        d = span(a, b)
        if d.size:
            total += np.median(d)
            print(f"{a:>8} -> {b:<12} median {np.median(d):6.0f}  mean {d.mean():7.1f}  p90 {np.percentile(d, 90):6.0f} cycles")
    print(f"sum of the medians: {total:.0f} cycles per warp-step")
    # phase between blocks that shared an SM from the start (the first wave: blocks 0 .. 3 x 148 - 1 all start together)
    by_sm = {}
    for b in range(len(s)):
        by_sm.setdefault(int(smid[b]), []).append(b)
    ph, lag = [], []
    for sm, bl in by_sm.items():
        bl = sorted(bl, key=lambda b: s[b, 0, 0, 0])[:3]
        if len(bl) < 2:
            continue
        for w in range(WARPS):
            per = np.median(np.diff(s[bl[0], w, :, 0]))
            for b in bl[1:]:
                d = float(np.median(s[b, w, :, 0] - s[bl[0], w, :, 0]))
                lag.append(d)
                ph.append((d % per) / per)
    ph = np.array(ph)
    near = np.minimum(ph, 1 - ph)
    print(f"phase of warp w of co-resident blocks against the SM's first block: {len(ph)} pairs; distance from lockstep "
          f"(fraction of a step, 0 = lockstep, 0.5 = opposite): median {np.median(near):.3f}, p10 {np.percentile(near, 10):.3f}, "
          f"p90 {np.percentile(near, 90):.3f}; share within 0.05: {(near < 0.05).mean():.2f}")
    hist, edges = np.histogram(near, bins=10, range=(0, 0.5))
    print("  histogram (0 .. 0.5 in tenths):", " ".join(str(h) for h in hist))


if __name__ == "__main__":
    {"build": build, "run": run}[sys.argv[1]](sys.argv[2])
