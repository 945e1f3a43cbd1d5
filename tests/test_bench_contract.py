"""Tests of bench.py.  CPU: the reference arm runs without a GPU, prints exactly one JSON line on stdout and carries the
result keys (metric / value / unit / config / impl / cpu_baseline / e2e ...).  GPU: --steps sets the timed steps and
--dump-outputs is repeatable."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "stereo_pairs_per_sec" and d["unit"] == "pairs/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("kitti00_shape") and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def run_bench(B, steps, *extra):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3", "--batch", str(B),
                        "--pool", "4", "--no-cpu-baseline", *extra], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout)
    assert line["steps"] == steps and line["config"]["pairs_per_step_per_gpu"] == B
    return line


@pytest.mark.gpu
def test_steps_sets_the_timed_steps(built):
    """--steps K runs K batches in the timed region: twice the steps, twice the kernel launches counted there."""
    n2, n4 = run_bench(8, 2)["gpu_launches"], run_bench(8, 4)["gpu_launches"]
    assert n2 > 0 and n4 == 2 * n2, (n2, n4)


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(built, tmp_path):
    """--dump-outputs: two runs with the same arguments write the same float32 / float64 arrays (at most 64 MB), so that
    two builds of the project can be compared output for output."""
    B = 8
    dumps = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        run_bench(B, 2, "--dump-outputs", str(d))
        dumps.append({f.stem: np.load(f) for f in sorted(d.glob("*.npy"))})
    a, b = dumps
    assert a.keys() == b.keys() and {"result_DT", "result_status", "device_poses", "features_pt_P", "features_ldesc"} <= a.keys()
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert a["result_DT"].shape == (B, 4, 4) and np.array_equal(a["device_poses"], a["result_DT"].reshape(B, 16))
    assert a["features_n_pt"].sum() == len(a["features_pt_P"]) > 0
