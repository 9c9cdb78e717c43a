"""bench.py contract pieces that can run without a GPU: the reference arm
(CPU port of the reference path) prints one JSON line with the agreed keys,
the B200 arm refuses to run (no CPU fallback) on a GPU-less box, and the
--dump-outputs writer keeps a fixed, bounded sample."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "3"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "transpose_GiB_per_s" and d["unit"] == "GiB/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["value"] > 0
    assert d["config"]["round_trip_bit_exact"] is True
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GiB/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}


def test_b200_arm_has_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0
    assert "no CPU fallback" in (out.stderr + out.stdout)


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0
    assert "--steps must be at least 1" in out.stderr


def test_dump_outputs_fixed_sample_within_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 48000)

    class U:
        def __init__(self, data):
            self.data = data
    big = U(torch.randn(40, 50, 3, dtype=torch.complex128, generator=torch.Generator().manual_seed(1)))
    small = U(torch.arange(24, dtype=torch.float32).reshape(2, 3, 4))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), [("big", big), ("small", small)], 0, 1, torch)
    a_big, b_big = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a_big.dtype == np.float64 and a_big.shape == (48000 // (2 * 16), 2)
    assert np.array_equal(a_big, b_big)
    # every sampled row is one element of the array, in memory order
    full = torch.view_as_real(big.data.reshape(-1)).numpy()
    pos = {v: i for i, v in enumerate(full[:, 0].tolist())}
    idx = [pos[v] for v in a_big[:, 0].tolist()]
    assert idx == sorted(set(idx)) and np.array_equal(full[idx], a_big)
    a_small = np.load(tmp_path / "a" / "small.npy")
    assert a_small.dtype == np.float32 and np.array_equal(a_small, np.arange(24, dtype=np.float32))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 48000 + 2 * 256
