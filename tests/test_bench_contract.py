"""CPU: the `bench.py --impl reference` arm (the reference algorithm = oracle port on the host cores) prints ONE JSON
line with the keys the driver's contract names; the product arm refuses to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, STEP_B200_CPU_THREADS=str(min(os.cpu_count() or 1, 16)))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("STEP fwd+bwd samples/sec") and d["value"] > 0 and d["n_gpus"] == 1
    assert d["steps"] == 1 and d["warmup"] == 0 and d["scaling"] == "weak" and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    # the reference's torch modules as restated by oracle/step_oracle.py (checked against the reference's golden outputs)
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_product_arm_needs_a_gpu():
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
