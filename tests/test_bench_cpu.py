"""bench.py host logic that the driver's contract depends on (no GPU): config table, workload accounting, the source hash that
stamps committed ncu captures, and the reference arm's JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_accounting_and_configs():
    sys.path.insert(0, ROOT)
    import bench
    assert set(bench.CONFIGS) == {"c2", "c3", "c4", "c5"}
    assert bench.tiles_1d(1024) == [576, 576] and bench.tiles_1d(576) == [576] and bench.tiles_1d(720) == [576, 272]
    assert bench.tiles_1d(1280) == [576, 576, 384]                      # 720p: 2 x 3 ragged tiles (SURVEY section 8d)
    # c2: one chunk x two 576x576 tiles; c4: 8 chunks of 17 frames x 6 tiles
    assert bench.workload_pixels(17, 576, 1024) == 17 * 576 * (576 + 576)
    assert bench.workload_pixels(129, 720, 1280) == 8 * 17 * (576 + 272) * (576 + 576 + 384)
    assert bench.workload_pixels(17, 256, 256, batch=32) == 32 * 17 * 256 * 256
    h = bench.source_hash()
    assert len(h) == 16 and h == bench.source_hash()
    assert bench.sample_shape(1)[3] == 192 and bench.sample_shape(23)[3] == 128 and bench.sample_shape(40)[3] == 96


def test_dump_outputs_writes_float32_within_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    assert 2 * bench.DUMP_MAX_ELEMS * 4 <= 64 << 20                              # latent + recon as float32 <= 64 MB
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 1000)
    small = torch.randn(2, 3, 4, dtype=torch.float16)
    big = torch.arange(5000, dtype=torch.bfloat16)
    info = bench.dump_outputs(str(tmp_path / "out"), {"latent": small, "recon": big})
    assert info == {"latent": {"shape": [2, 3, 4], "stored": 24}, "recon": {"shape": [5000], "stored": 1000}}
    a, b = np.load(tmp_path / "out" / "latent.npy"), np.load(tmp_path / "out" / "recon.npy")
    assert a.dtype == np.float32 and np.array_equal(a, small.float().numpy())   # small arrays whole and exact
    assert b.dtype == np.float32 and b.shape == (1000,) and np.all(np.diff(b) >= 0) and set(b) <= set(big.float().numpy())
    assert np.array_equal(b, bench.dump_array(big))                              # the sample is fixed


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--height", "64", "--width", "64", "--frames", "5"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["value"] > 0
