"""Developer helper (GPU box): small launches of every round-2 kernel for compute-sanitizer.
usage: compute-sanitizer --tool racecheck python tools/sanitize_case.py"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from optistate_b200 import kf_batch  # noqa: E402
from optistate_b200.mpc import WarmStart, mpc_forces  # noqa: E402
from optistate_b200.synth import make_streams  # noqa: E402
from tests import mpc_cases  # noqa: E402

S, T, N = 64, 12, 64 * 6 + 64  # seven members per stream: two groups of warps per tile, the second one ragged
st = make_streams(range(S), T)
q, r = bench.mc_noise(0, N, S)
for dt in (torch.float64, torch.float32):
    d = {k: torch.from_numpy(v).to("cuda", dt) for k, v in st.items()}
    nominal = kf_batch(d["imu"], d["p"], d["dp"], d["contact"], d["f"], dtype=dt, outputs=("x_steps",)).x_steps
    for structure in ("auto", "full"):
        for outputs in (("summary",), ("x_steps", "p_trace"), ("x_final", "p_world_steps")):
            kw = dict(truth=d["truth"], nominal=nominal) if outputs == ("summary",) else {}
            res = kf_batch(d["imu"], d["p"], d["dp"], d["contact"], d["f"], Q=q, R=r, n_traj=N, dtype=dt, outputs=outputs, structure=structure, **kw)
    torch.cuda.synchronize()
    print("streamed kernels", dt, res.algo, "ok", flush=True)
n = 96
x, ref, p, c = mpc_cases.batch(n, seed=2)
trot = np.where((np.arange(n) % 2 == 0)[None, :], np.array([1.0, 0, 0, 1])[:, None], np.array([0, 1.0, 1, 0])[:, None])
warm = WarmStart(n)
for _ in range(2):
    f1, s1 = mpc_forces(x, ref, p, trot, warm=warm)                      # dual active set, one warp (cold, then warm)
f2, s2 = mpc_forces(x, ref, p, trot, solver="interior_point")            # shared-memory interior point
warm4 = WarmStart(n)
for _ in range(2):
    f3, s3 = mpc_forces(x, ref, p, c, warm=warm4)                        # all contact patterns: two warps per problem
torch.cuda.synchronize()
print("mpc kernels ok; flags", int((s1 & 7).max()), int((s2 & 7).max()), int((s3 & 7).max()), "agreement", float((f1 - f2).abs().max()), flush=True)
