"""bench.py's reference arm runs on the CPU: the JSON line it prints is checked against the driver's contract here (the GPU arm
prints the same keys plus roofline / clocks / parity, checked on the GPU box by the bench run itself)."""
import json
import subprocess
import sys

import numpy as np

from conftest import ROOT


def test_reference_arm_line(tmp_path):
    from oracle.bindings import REF_SO
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-trials-per-point", "2",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "decoded_frames_per_s" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["steps"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["value"] == d["value"] and cb["cores"] >= 1 and "2 trials per QBER point" in cb["sample"]
    assert cb["kind"] == ("reference" if REF_SO.exists() else "port")
    assert d["config"]["workload"].startswith("configs[1]") and len(d["config"]["qber_grid"]) == 9
    assert [round(x["fer"]) for x in d["per_qber"]] == [0, 0, 0, 0, 0, 0, 1, 1, 1]  # 0.03 ... 0.08 converge, 0.09 ... 0.11 do not
    it, flags = np.load(tmp_path / "iterations.npy"), np.load(tmp_path / "result_flags.npy")
    assert it.dtype == flags.dtype == np.float32 and it.shape == flags.shape == (9, 2)
    assert (1.0 - (flags == 3).mean(1)).tolist() == [x["fer"] for x in d["per_qber"]]
    assert np.load(tmp_path / "point_stats.npy")[:, -2].tolist() == [2.0] * 9  # trials per point


def test_reference_arm_other_ranks_exit_quietly():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True, cwd=ROOT, env=env, timeout=120)
    assert p.returncode == 0 and p.stdout.strip() == ""
