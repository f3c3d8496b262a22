"""CPU-side tests of bench.py's host logic: the executed-flop / traffic figures are READ from the committed ncu summaries (not
typed in), job shapes for weak / strong scaling, the noise law, the clock sampler without a GPU, and the reference arm."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _bench(*extra, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=timeout)
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_executed_flops_and_traffic_come_from_the_committed_ncu_summaries():
    """Round-1 summaries (full 78-entry kernels): the parser reproduces the figures round 1 had typed into bench.py
    (1135 DFMA x 2 + 321 DMUL + 99 DADD = 2,690; FP32 pair kernel 2,562 per trajectory; 2.724 + 0.433 GB of DRAM traffic)."""
    f64 = bench.kernel_profile("f64", "full", tags=("r1",))
    assert f64["flops_executed"] == 2 * 1135 + 321 + 99 and f64["fp_instructions_per_thread_step"] == 1555 and f64["lanes"] == 1
    assert abs(f64["traffic_bytes"] - (2.723607e9 + 433.020928e6)) < 1e3 and f64["grid"] == 8192
    f32 = bench.kernel_profile("f32", "full", tags=("r1",))
    assert f32["lanes"] == 2 and f32["flops_executed"] == (2 * 2 * 1051 + 2 * 302 + 2 * 85 + 2 * 54 + 30 + 8) / 2
    # a capture of ANOTHER instantiation is never used: round 1 has no decoupled-group kernel
    assert bench.kernel_profile("f64", "auto", tags=("r1",)) is None


def test_current_profiles_describe_the_kernels_that_are_built():
    """Every r2 hot-loop summary must name an instantiation that exists in the built library, and its executed FP count must
    not exceed the static count of that kernel's time loop (tools/sass_loop.py; the static loop also holds the rare slow paths): an edit of the kernel that is not followed by
    a new capture shows up here."""
    import glob

    from optistate_b200 import _build
    from tools import sass_loop

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r2_ncu_bench_kernel_*_hotloop.txt")))
    for f in files:
        tag = os.path.basename(f).split("_ncu_bench_kernel_")[1].replace("_hotloop.txt", "")
        dtype, structure = tag.split("_")[0], ("full" if tag.endswith("_full") else "auto")
        prof = bench.kernel_profile(dtype, structure, tags=("r2",))
        assert prof is not None, f
        real = {"double": "d", "float": "f", "okf::F2": "NS_2F2E"}[prof["kernel"].split("<")[1].split(",")[0].strip()]
        mangled = f"kf_seq_tma_kernelI{real}Lb1ELi0ELb0ELb{1 if structure == 'auto' else 0}ELi0EE"  # ..., kW = 0: the throughput geometry
        hist = sass_loop.loop_histogram(_build.KF_LIB, mangled)
        assert len(hist) == 1, (mangled, list(hist))
        h, _ = next(iter(hist.values()))
        _, n_static = sass_loop.flops(h)
        assert 0.5 * n_static <= prof["fp_instructions_per_thread_step"] <= n_static, (f, n_static, prof["fp_instructions_per_thread_step"])


def test_job_shapes_and_noise_law():
    class A:
        traj_total, traj_per_gpu = 0, 1 << 20
    assert bench.job_shape(A, 8, 3) == (8 << 20, 3 << 20, 1 << 20, "weak")
    A.traj_total = (1 << 24) + 3
    tot = 0
    for rk in range(8):
        n_total, first, n_local, scaling = bench.job_shape(A, 8, rk)
        assert scaling == "strong" and first == tot and n_total == A.traj_total
        tot += n_local
    assert tot == A.traj_total
    # the noise is a function of the member id: any shard draws what the whole job would draw
    q, r = bench.mc_noise(0, 70000, 1024)
    q2, r2 = bench.mc_noise(65000, 5000, 1024)
    assert np.array_equal(q[:, 65000:], q2) and np.array_equal(r[:, 65000:], r2)
    assert np.array_equal(q[:, :1024], np.repeat(bench.Q_DIAG[:, None], 1024, 1)) and (q[:, 1024:] != bench.Q_DIAG[:, None]).all()
    assert 10 ** -0.5 <= (r / 0.01).min() and (r / 0.01).max() <= 10 ** 0.5


def test_parity_sample_is_zero_against_itself_and_sees_a_wrong_member():
    from oracle import c_oracle
    from optistate_b200.synth import make_streams

    st = make_streams(range(8), 60)
    idx = np.array([0, 3, 7, 3], np.int32)
    q, r = bench.mc_noise(0, 4, 2)
    ref = c_oracle.run(st, 4, Q=q, R=r, stream_index=idx, want=("x_steps", "P_final", "nis_steps", "p_trace_steps", "k_gain_steps"))
    nominal = c_oracle.run(st, want=("x_steps",))["x_steps"]
    sm = np.zeros((52, 4))
    x = ref["x_steps"]
    sm[0:12], sm[12:24] = x[-1], ref["P_final"][::13]
    sm[24:36] = np.sqrt(((x - st["truth"][:, :, idx]) ** 2).mean(axis=0))
    sm[36:48] = np.sqrt(((x - nominal[:, :, idx]) ** 2).mean(axis=0))
    sm[48], sm[49], sm[50], sm[51] = ref["nis_steps"].mean(axis=0), ref["p_trace_steps"][-1], ref["k_gain_steps"][-1], np.sqrt(ref["nis_steps"].max(axis=0))
    e = bench.parity_sample(st, q, r, idx, sm, nominal)
    assert e["n"] == 4 and max(v for k, v in e.items() if k.startswith("max_rel_")) == 0.0
    sm[5, 2] *= 1.0 + 1e-6
    assert bench.parity_sample(st, q, r, idx, sm, nominal)["max_rel_x"] > 1e-7


def test_parity_sample_with_ten_and_twelve_members_reads_the_noise_per_trajectory():
    """A sample of exactly 10 (12) members hands the oracle a [10, 10] R ([12, 12] Q): it must still be read as per-trajectory
    diagonals, not as one shared dense matrix (this made the full-size FP64 test fail on its first GPU run)."""
    from oracle import c_oracle
    from optistate_b200.synth import make_streams

    st = make_streams(range(4), 40)
    for n in (10, 12):
        idx = (np.arange(n) % 4).astype(np.int32)
        q, r = bench.mc_noise(4, n, 4)
        batch = c_oracle.run(st, n, Q=q, R=r, stream_index=idx, noise_per_traj=True, want=("x_final",))["x_final"]
        for k in range(n):
            one = c_oracle.run(st, 1, Q=q[:, [k]], R=r[:, [k]], stream_index=idx[k:k + 1], want=("x_final",))["x_final"]
            assert np.array_equal(one[:, 0], batch[:, k]), (n, k)
        sm = np.zeros((52, n))
        sm[0:12] = batch
        assert bench.parity_sample(st, q, r, idx, sm)["max_rel_x"] == 0.0


def test_dump_sample_is_fixed_and_fits_the_dump_budget():
    assert np.array_equal(bench.dump_members(100), np.arange(100))
    m = bench.dump_members(1 << 20)
    assert m.size == bench.DUMP_MEMBERS and np.array_equal(m, bench.dump_members(1 << 20))
    assert (np.diff(m) > 0).all() and 0 <= m[0] and m[-1] < 1 << 20
    assert (52 + 3) * 8 * m.size <= 64 << 20  # FP64 summary columns + member ids + status words and their member ids


def test_clock_sampler_survives_a_box_without_gpu_or_nvml():
    with bench.ClockSampler(0, period=0.01) as c:
        pass
    s = c.summary()
    assert set(s) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples", "how"}


def test_bench_reference_arm_line(tmp_path):
    d = _bench("--impl", "reference", "--steps", "1", "--warmup", "1", "--T", "50", "--dump-outputs", str(tmp_path))
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    # --dump-outputs: the final states of the last timed step, as the C oracle computes them for the same members and noise
    x, members = np.load(tmp_path / "x_final.npy"), np.load(tmp_path / "members.npy")
    assert sorted(os.listdir(tmp_path)) == ["members.npy", "x_final.npy"] and x.dtype == np.float64 and x.shape == (12, members.size)
    from oracle import c_oracle
    from optistate_b200.synth import make_streams

    n = int(members.max()) + 1
    q, r = bench.mc_noise(0, n, 64)
    want = c_oracle.run(make_streams(range(64), 50), n, Q=q, R=r, want=("x_final",))["x_final"]
    assert np.array_equal(x, want[:, members.astype(np.int64)])
    if os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "kalman_filter", "kalman_filter.py")) or os.path.isdir("/root/reference"):
        assert d["cpu_baseline"]["reference_class_steps_per_s_1core"] > 100  # the unmodified reference class, timed on this box
