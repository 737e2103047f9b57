"""The JSON line of `bench.py --impl reference` (the arm that runs on host cores, so it can be checked without a GPU)
carries every key of the driver's contract; under torchrun only rank 0 prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def _run(extra, env=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3",
           "--ref-budget-s", "2"] + extra
    return subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)


def test_reference_arm_line_has_the_contract_keys():
    res = _run(["--threads", "2"])
    assert res.returncode == 0, res.stderr
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert KEYS <= set(d), KEYS - set(d)
    assert d["impl"] == "reference" and d["unit"] == "MB/s" and d["higher_is_better"] is True and d["warmup"] >= 3
    assert d["metric"].startswith("protected-kernel throughput (MB/s voted output)") and d["value"] > 0
    assert d["config"]["workload"].startswith("sha256 TMR, 2^20 x 64-byte messages")
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] == 2 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_print_nothing():
    res = _run([], env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert res.returncode == 0 and not [ln for ln in res.stdout.splitlines() if ln.startswith("{")]


def test_both_arms_print_the_same_config_object():
    """VERDICT r01: `same_config` was false because the arms' config dicts carried different keys.  config is now a pure
    function of (workload, GPU count) that both arms call."""
    sys.path.insert(0, ROOT)
    import bench
    res = _run(["--threads", "2", "--gpus", "1"])
    d = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][0])
    assert d["config"] == bench.config_for("sha256", 1)
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": config_for(wl, ') == 2          # the reference arm and the GPU arm, nothing hand-written
    for wl in bench.WORKLOAD_NAMES:
        assert bench.config_for(wl, 8)["parallelism"] == "shard8" and bench.config_for(wl, 8)["workload"] == bench.WORKLOAD_NAMES[wl]


def test_dumped_output_sample_is_exact_seeded_and_bounded(tmp_path):
    """--dump-outputs: the same units are sampled on every run, their words are widened without loss, and the files of
    every workload together stay within the size bound."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    n = 3 * bench.DUMP_UNITS
    out = torch.from_numpy(np.random.default_rng(1).integers(0, 256, n * 32, dtype=np.uint8))
    vals, units = bench.output_sample(torch, out, n, 0, "sha256")
    again, units2 = bench.output_sample(torch, out, n, 0, "sha256")
    assert vals.dtype == np.float64 and vals.shape == (bench.DUMP_UNITS, 8) and np.array_equal(units, units2)
    assert np.array_equal(vals, again)
    assert np.array_equal(vals, out.numpy().view("<u4").reshape(n, 8)[units.astype(np.int64)])
    c = torch.randn(100)
    vals, units = bench.output_sample(torch, c, 100, 7, "gemm")
    assert np.array_equal(vals[:, 0], c.numpy()) and units[0] == 7
    words = {wl: bench.OUT_B[wl] // np.dtype(w).itemsize for wl, w in bench.DUMP_WORD.items()}
    total = sum(bench.DUMP_UNITS * (words[wl] * (8 if w == "<u4" else 4) + 8) for wl, w in bench.DUMP_WORD.items())
    assert total <= bench.DUMP_MAX_BYTES
    bench.write_dump(str(tmp_path), {"gemm": vals})
    assert np.array_equal(np.load(tmp_path / "gemm.npy"), vals)


def test_reference_arm_reports_the_median_of_individually_timed_steps():
    res = _run(["--threads", "2", "--workload", "crc16"])
    d = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][0])
    assert "median" in d["cpu_baseline"]["sample"] and "pinned" in d["cpu_baseline"]["sample"] and d["cpu_baseline"]["spread"] >= 1.0
