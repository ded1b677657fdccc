"""bench.py's output contract: the JSON line (keys, units, types) on the reference arm, which runs on CPU, and the arrays
`--dump-outputs` writes on the GPU arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-batch", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images_per_sec" and d["unit"] == "img/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_only_rank0_prints():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_world2_is_the_gloo_ddp_syncbn_loop():
    """at N > 1 the reference arm times the reference's DISTRIBUTED loop on the host: N gloo ranks (BASELINE.md §3 rows 3-4)"""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
                          "--cpu-batch", "2"], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["n_gpus"] == 2 and "2 gloo ranks" in d["cpu_baseline"]["sample"] and "2 CPU ranks" in d["config"]["workload"]
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-extras",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 2
    loss, items, logits = (np.load(tmp_path / f"{n}.npy") for n in ("loss", "loss_items", "logits"))
    assert loss.dtype == items.dtype == logits.dtype == np.float32
    assert loss.shape == () and items.shape == (8,) and logits.shape == (16, 1, 320, 320)
    assert loss == items[2] and items[7] == logits.size and np.isfinite(logits).all()
