"""The JSON line bench.py prints is a contract with the driver: check the keys on the committed round-2 lines (produced
on B200 by the commands named in profiles/INDEX.md) and on a reference-arm line produced here, on the host cores."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def _check_common(d, cpu_baseline=True):
    keys = BASE_KEYS if cpu_baseline else BASE_KEYS - {"cpu_baseline"}  # (the CPU baseline is an N = 1 item)
    assert keys <= set(d), keys - set(d)
    assert d["metric"] == "fp8_attn_fwd_tflops" and d["unit"] == "TFLOP/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None  # BASELINE.md publishes no number for this metric
    assert "workload" in d["config"] and "model" not in d["config"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    if cpu_baseline:
        assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])


@pytest.mark.parametrize("name", ["r02_bench_c2_driver.json", "r02_bench_c2.json", "r02_bench_c3.json"])
def test_committed_gpu_lines_carry_the_contract(name):
    d = json.load(open(os.path.join(ROOT, "profiles", name)))
    _check_common(d)
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert r["bound"] == "tensor" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["achieved"] >= d["value"] * 0.999  # the kernel alone is never slower than the step it is part of
    assert r["achieved"] <= r["peak"]
    assert d["gpu_launches"] >= 2 * d["steps"]  # quantiser + attention per step
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["e2e"]["value"] < d["value"]  # host buffers, copies inside the timed region
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["dtype"].startswith("fp8_e4m3") and d["data"].startswith("synthetic")


@pytest.mark.parametrize("n", [2, 4, 8])
def test_committed_scaling_lines_carry_the_sequence_sharded_block(n):
    d = json.load(open(os.path.join(ROOT, "profiles", f"r02_bench_c2_n{n}.json")))
    _check_common(d, cpu_baseline=False)
    assert d["n_gpus"] == n and d["scaling"] == "weak"
    s = d["seq_sharded"]
    assert s["scaling"] == "strong" and s["n_gpus"] == n
    assert s["strong_scaling_efficiency"] >= 0.85  # the round-1 review's bar for the C4 curve
    acc = s["accuracy"]
    for mode in ("16bit", "fp8_hilo"):  # the stated bounds, on the line itself
        assert acc[mode]["cos_sim"] >= 0.999 and acc[mode]["max_abs_over_row_rms"] <= 0.02
    assert acc["fp8"]["cos_sim"] >= 0.999  # (single e4m3 P: cosine bound only - why it is opt-in)


def test_reference_arm_runs_on_the_host_cores_with_the_same_config():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    _check_common(d)
    assert d["impl"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["steps"] == 1 and "median of 1 runs" in d["cpu_baseline"]["sample"]  # --steps is the number of timed runs
    ours = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_c2_driver.json")))
    assert set(d["config"]) == set(ours["config"]) and d["config"]["workload"] == ours["config"]["workload"]


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs"]])
def test_bench_rejects_what_it_cannot_honour(argv, tmp_path):
    if argv[-1] == "--dump-outputs":
        argv = argv + [str(tmp_path / "dump")]
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 2 and out.stdout == "", out.stderr[-2000:]
    assert not os.path.exists(tmp_path / "dump")


def test_dump_outputs_writes_float32_whole_or_a_fixed_sample_of_rows(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench

    out = torch.randn(2, 3, 50, 64, generator=torch.Generator().manual_seed(0)).to(torch.bfloat16)
    bench.dump_outputs(str(tmp_path / "whole"), out)
    whole = np.load(tmp_path / "whole" / "out.npy")
    assert whole.dtype == np.float32 and np.array_equal(whole, out.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 4 * 64 * 10)  # room for 10 rows of D = 64
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), out)
    a, b = np.load(tmp_path / "a" / "out.npy"), np.load(tmp_path / "b" / "out.npy")
    assert a.dtype == np.float32 and a.shape == (10, 64) and np.array_equal(a, b)
    rows = whole.reshape(-1, 64)
    idx = [int(np.flatnonzero((rows == r).all(1))[0]) for r in a]
    assert idx == sorted(set(idx))  # distinct rows of the output, in their order
