"""Harness tests (bench.py's measurement contract).  The file name sorts LAST on purpose: a tooling failure here must never
hide a parity test under `pytest -x` (round 1 lost the seven fused-all-gather tests that way)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*extra, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=timeout)
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_bench_native_arm_prints_the_contract_line():
    """bench.py on a small workload: every key of the measurement contract is present and self-consistent."""
    d = _bench("--steps", "2", "--warmup", "3", "--traj-per-gpu", "8192", "--T", "60", "--streams", "128", "--no-cpu-baseline", "--no-secondary")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "e2e", "gpu_launches", "clocks", "roofline", "parity_sample"):
        assert k in d, k
    assert d["metric"] == "kf_trajectory_steps_per_sec" and d["unit"] == "trajectory-steps/s" and d["n_gpus"] == 1 and d["dtype"] == "f64"
    assert d["steps"] == 2 and d["warmup"] == 3 and d["higher_is_better"] is True and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["scaling"] == "weak" and d["config"]["trajectories_total"] == 8192
    assert abs(d["value"] - 8192 * 60 * 2 / (d["ms_per_step"] * 2e-3)) < 1e-6 * d["value"]
    assert d["gpu_launches"] >= 2 * 2  # measurement pre-pass + filter kernel per step
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] == 52 * 8192 * 8
    r = d["roofline"]
    assert r["bound"] == "fma" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and r["peak"] > 10
    assert abs(r["frac_algorithmic"] - r["achieved_algorithmic"] / r["peak"]) < 1e-12
    assert r["measured_fma_peak_tflops"] > 0.9 * r["theoretical_peak_at_sampled_clock_tflops"]  # the probe saturates the FP64 pipe
    assert d["status_nonzero_trajectories"] == 0
    # the short region still has its two synchronous clock readings (round 1: a 200 ms poll saw none)
    assert d["clocks"]["sm_mhz"] is not None and d["clocks"]["samples"] >= 2 and d["clocks"]["sm_max_mhz"] >= d["clocks"]["sm_mhz"]
    ps = d["parity_sample"]
    assert ps["ok"] and ps["n"] >= 8 and ps["max_rel_x"] < 1e-9 and ps["max_rel_p"] < 1e-9


def test_bench_strong_scaling_mode_and_full_covariance_structure():
    """--traj-total shards a fixed job (BASELINE configs[3] is --traj-total 16777216); --structure full times the 78-entry kernel."""
    d = _bench("--steps", "1", "--warmup", "3", "--traj-total", "4096", "--T", "50", "--streams", "64", "--no-cpu-baseline", "--no-secondary",
               "--no-e2e", "--structure", "full")
    assert d["scaling"] == "strong" and d["config"]["trajectories_total"] == 4096 and d["parity_sample"]["ok"]
    assert "78" in d["config"]["covariance_structure"]


def test_bench_dump_outputs_are_the_oracles_and_the_same_in_every_run(tmp_path):
    """--dump-outputs writes the summaries and status words the timed path returned in its last step: the dumped columns are
    those the C oracle computes for the listed members, and two runs with the same arguments dump identical arrays."""
    import bench
    from oracle import c_oracle
    from optistate_b200.synth import make_streams

    args = ("--steps", "2", "--warmup", "1", "--traj-per-gpu", "4096", "--T", "50", "--streams", "64", "--no-cpu-baseline", "--no-secondary", "--no-e2e")
    for run in ("a", "b"):
        d = _bench(*args, "--dump-outputs", str(tmp_path / run))
        assert d["steps"] == 2 and d["parity_sample"]["ok"]
    names = ("members", "status", "status_members", "summary")
    a, b = ({k: np.load(tmp_path / run / f"{k}.npy") for k in names} for run in ("a", "b"))
    assert sorted(os.listdir(tmp_path / "a")) == [k + ".npy" for k in names]
    assert a["summary"].shape == (52, 4096) and a["summary"].dtype == np.float64
    assert np.array_equal(a["members"], np.arange(4096)) and np.array_equal(a["status_members"], a["members"]) and not a["status"].any()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    # columns of members other than those bench.py's parity sample picks, against the oracle on the same streams and noise
    st = make_streams(range(64), 50)
    pick = np.array([1, 2, 63, 64, 65, 1000, 2047, 3001, 4094])
    qs = np.concatenate([bench.mc_noise(int(m), 1, 64)[0] for m in pick], axis=1)
    rs = np.concatenate([bench.mc_noise(int(m), 1, 64)[1] for m in pick], axis=1)
    nominal = c_oracle.run(st, want=("x_steps",))["x_steps"]
    cols = a["summary"][:, np.searchsorted(a["members"], pick)]
    e = bench.parity_sample(st, qs, rs, (pick % 64).astype(np.int32), cols, nominal)
    assert max(v for k, v in e.items() if k.startswith("max_rel_") and k != "max_rel_dev") < 1e-9 and e["max_rel_dev"] < 1e-7, e
