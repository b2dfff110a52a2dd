"""CPU-only: the reference arm of bench.py (`--impl reference`: the compiled reference ODE, or the C port, on host
threads) prints one JSON line with the contract's keys. The GPU arm is exercised on the GPU box by the driver."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "poses/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_reference_arm_dumps_its_outputs(tmp_path):
    """--dump-outputs writes the verdicts of the last timed step as float .npy files, identical from run to run."""
    import numpy as np
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                            "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
    a, b = (np.load(tmp_path / d / "valid.npy") for d in ("a", "b"))
    assert a.dtype == np.float32 and a.shape == (200_000,) and 0 < a.sum() < len(a)
    assert np.array_equal(a, b)


def test_bench_metric_matches_baseline_json():
    b = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert "pose-validity checks/s" in src
    assert "pose" in json.dumps(b).lower()
