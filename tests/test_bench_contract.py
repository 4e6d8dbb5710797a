"""bench.py's reference arm runs on the host alone: check the JSON line it prints against the bench contract
(the GPU arm prints the same keys plus roofline / clocks / gpu_launches; it needs a B200 and is exercised by the driver)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=env, cwd=ROOT, timeout=900)


def test_reference_arm_json_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                   # exactly ONE JSON line
    j = json.loads(lines[0])
    assert j["impl"] == "reference"
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert j["metric"].split(" @")[0] in baseline["metric"]   # BASELINE.json's metric, not one of our own
    assert j["unit"] == "Mpixels/s" and j["higher_is_better"] is True and j["scaling"] == "weak"
    assert j["n_gpus"] == 1 and j["steps"] == 1 and j["warmup"] == 0
    assert j["value"] > 0 and j["ms_per_step"] > 0
    assert j["vs_baseline"] is None                           # BASELINE.md publishes no number for this metric
    assert j["data"] == "synthetic" and "workload" in j["config"] and "model" not in j["config"]
    cb = j["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == j["value"]
    e2e = j["e2e"]
    assert e2e["value"] == j["value"] and e2e["unit"] == j["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_stay_silent():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29591"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_is_refused_outside_the_gpu_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_step(tmp_path):
    """--dump-outputs: the four arrays the timed step returns, float32, within 64 MB; --steps sets the timed steps"""
    import numpy as np
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-extras", "--no-e2e",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert j["steps"] == 2 and j["gpu_launches"] == 2 * 2          # one fused forward + one fused backward per step
    files = sorted(p.name for p in tmp_path.iterdir())
    assert files == ["grad_flow.npy", "grad_logits.npy", "grad_source.npy", "out.npy"]
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    arrays = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
    assert arrays["grad_flow"].size == 16 * 2 * 256 * 256                 # small enough to be written whole
    assert arrays["out"].std() > 0 and arrays["grad_source"].std() > 0
