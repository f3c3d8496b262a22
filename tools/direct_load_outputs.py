"""Developer helper: every output tensor and status word of the direct-load SEQUENTIAL kernel (kf_seq_kernel, which a
stream_index selects) on a fixed set of seeded cases, saved to one file; `compare` checks two such files with torch.equal.  Run
`dump` in two source trees (say the parent of a change and the change, each built) and compare the files, to show that a
refactor of the kernel left its results bit for bit alone.

    python tools/direct_load_outputs.py dump OUT.pt [--root TREE]      (on a GPU; TREE: the tree whose build to import)
    python tools/direct_load_outputs.py compare A.pt B.pt

Cases: FP64 and FP32; structure "auto" and "full"; cov_model "mpc"; per-trajectory Q, R, x0 and a dense per-trajectory P0; the
summary with truth and nominal streams; every per-step output with ckpt_every; P_steps through kf_smooth and kf_smooth_full; a
ragged last block (N = 300 with 128-thread blocks), N = 0 and T = 0."""
import argparse
import os
import sys


def cases(torch, np, ob, synth):
    from optistate_b200.settings import INITIAL_PARAMS  # noqa: F401  (import check of the tree)

    S, T, N = 64, 120, 300
    st = synth.make_streams(range(700, 700 + S), T)
    q, r = synth.monte_carlo_noise(np.arange(N), np.full(12, 1e-3), np.full(10, 1e-2))
    idx = ((np.arange(N) * 7 + 3) % S).astype(np.int32)
    args = lambda s: (s["imu"], s["p"], s["dp"], s["contact"], s["f"])
    every = ("x_steps", "x_model_steps", "p_world_steps", "z_steps", "p_trace", "k_gain", "nis", "P_ckpt", "final", "summary")
    out = {}

    def put(name, res):
        for k, v in res.tensors.items():
            out[f"{name}/{k}"] = v.detach().cpu()
        out[f"{name}/status"] = res.status.detach().cpu()

    for dtype in (torch.float64, torch.float32):
        dn = "f64" if dtype == torch.float64 else "f32"
        kw = dict(Q=q, R=r, n_traj=N, dtype=dtype, stream_index=idx, ckpt_every=25, truth=st["truth"], nominal=0.5 * st["truth"])
        for structure in ("auto", "full"):
            a = ob.kf_batch(*args(st), structure=structure, outputs=every, **kw)
            put(f"{dn}/{structure}/all", a)
            put(f"{dn}/{structure}/summary_only", ob.kf_batch(*args(st), structure=structure, outputs=("summary",), **kw))
            put(f"{dn}/{structure}/truth_only", ob.kf_batch(*args(st), structure=structure, outputs=("summary", "x_steps"),
                                                            **dict(kw, nominal=None)))
            # per-trajectory x0 and a dense per-trajectory P0 (p0_kind 4), from the first run's final state
            put(f"{dn}/{structure}/x0_P0", ob.kf_batch(*args(st), structure=structure, x0=a.x_final, P0=a.P_final, p0_kind=4,
                                                       outputs=("final", "summary"), **kw))
        put(f"{dn}/mpc/all", ob.kf_batch(*args(st), cov_model="mpc", body_ref=st["truth"], outputs=every, **kw))
        put(f"{dn}/mpc/nosum", ob.kf_batch(*args(st), cov_model="mpc", body_ref=st["truth"], outputs=("x_steps", "final"),
                                           **dict(kw, truth=None, nominal=None)))
        sm = dict(Q=q, R=r, n_traj=N, dtype=dtype, stream_index=idx)
        put(f"{dn}/smooth", ob.kf_smooth(*args(st), outputs=("x_smooth", "var_smooth", "x_steps", "final"), **sm))
        put(f"{dn}/smooth_full", ob.kf_smooth_full(*args(st), outputs=("x_smooth", "var_smooth", "x_steps", "final"), **sm))
        put(f"{dn}/smooth_full_mpc", ob.kf_smooth_full(*args(st), cov_model="mpc", body_ref=st["truth"],
                                                       outputs=("x_smooth", "var_smooth", "final"), **sm))
        # N = 0 and T = 0
        put(f"{dn}/n0", ob.kf_batch(*args(st), Q=q[:, :0], R=r[:, :0], n_traj=0, dtype=dtype, stream_index=idx[:0],
                                    outputs=("x_steps", "final", "summary"), truth=st["truth"]))
        s0 = {k: v[:0] for k, v in st.items()}
        put(f"{dn}/t0", ob.kf_batch(*args(s0), **dict(kw, truth=s0["truth"], nominal=None, ckpt_every=0),
                                    outputs=("x_steps", "final", "summary")))
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=("dump", "compare"))
    ap.add_argument("files", nargs="+")
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    a = ap.parse_args()
    import torch

    if a.mode == "compare":
        x, y = torch.load(a.files[0]), torch.load(a.files[1])
        bad = [k for k in x if k not in y or x[k].dtype != y[k].dtype or x[k].shape != y[k].shape or not torch.equal(x[k], y[k])]
        bad += [k for k in y if k not in x]
        n = sum(v.numel() for v in x.values())
        print(f"{len(x)} tensors ({n} values): {len(x) - len(bad)} bit-identical, {len(bad)} differ")
        for k in bad:
            print("  differs:", k)
        sys.exit(1 if bad else 0)
    sys.path.insert(0, os.path.abspath(a.root))
    import numpy as np

    import optistate_b200 as ob
    from optistate_b200 import synth

    assert os.path.abspath(ob.__file__).startswith(os.path.abspath(a.root)), ob.__file__
    out = cases(torch, np, ob, synth)
    torch.save(out, a.files[0])
    print(f"{a.files[0]}: {len(out)} tensors from {os.path.abspath(a.root)}")


if __name__ == "__main__":
    main()
