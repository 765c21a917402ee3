"""GPU: `bench.py --dump-outputs` writes what the last timed step computed, and the same arguments give the same outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--only-resident",
                          "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["gpu_launches"] > 0
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_the_last_step_and_repeat(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    a, b = _bench_dump(tmp_path / "a"), _bench_dump(tmp_path / "b")
    assert sorted(a) == sorted(b)
    n, B, _ = bench.WORKLOADS["METR-LA"]
    assert a["y_hat"].shape == (B, 12, n, 1) and a["theta"].shape == a["adj_knn"].shape == (B, n, n)
    assert a["loss"].shape == () and a["gsl_coefficient"] == 1.0
    assert a["grad.backend.start_conv.weight"].shape == (32, 2, 1, 1)
    assert a["grad.discrete_graph_learning.fc.weight"].shape == (bench.DUMP_MAX_ELEMS,)      # sampled
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        if k.startswith("grad."):      # backward kernels accumulate with atomics: summation order varies run to run
            assert np.abs(v - b[k]).max() <= 2e-5 * np.abs(v).max(), k
        else:
            assert np.array_equal(v, b[k]), k
