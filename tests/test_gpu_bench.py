"""bench.py on the GPU at a tiny size: one JSON line whose step count is the one asked for, and --dump-outputs writes
the same arrays on two runs with the same arguments (seeded weights and inputs, deterministic engine)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0",
                        "--frames", "5", "--height", "64", "--width", "96", "--no-cpu-baseline", "--no-torch-baseline",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_bench_dump_outputs_are_reproducible(tmp_path):
    a, b = _run(tmp_path / "a"), _run(tmp_path / "b")
    assert a["steps"] == 2 and a["value"] > 0
    assert a["dumped"] == {"latent": {"shape": [1, 4, 2, 8, 12], "stored": 768},
                           "recon": {"shape": [1, 3, 5, 64, 96], "stored": 92160}}
    for name in ("latent", "recon"):
        x, y = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert x.dtype == np.float32 and list(x.shape) == a["dumped"][name]["shape"]
        assert np.isfinite(x).all() and np.array_equal(x, y), name
