"""CPU: bench.py's --dump-outputs writer and its argument checks (both act before any device work)."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_float32_and_float64(tmp_path):
    x0 = torch.arange(2 * 3 * 4, dtype=torch.float16).reshape(2, 3, 4)
    bench.dump_outputs(str(tmp_path), {"x0": x0, "loss": torch.tensor([0.25], dtype=torch.float64)})
    a, loss = np.load(tmp_path / "x0.npy"), np.load(tmp_path / "loss.npy")
    assert a.dtype == np.float32 and np.array_equal(a, x0.float().numpy())
    assert loss.dtype == np.float64 and loss.tolist() == [0.25]


def test_dump_outputs_over_budget_keeps_the_same_seeded_rows(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1000)
    x0 = torch.arange(100 * 3 * 4, dtype=torch.float32).reshape(100, 3, 4)
    loss = torch.tensor([0.5], dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"x0": x0, "loss": loss})
    a, b = np.load(tmp_path / "a" / "x0.npy"), np.load(tmp_path / "b" / "x0.npy")
    assert np.array_equal(a, b)
    assert a.nbytes + np.load(tmp_path / "a" / "loss.npy").nbytes <= 1000
    rows = a[:, 0, 0].astype(np.int64) // 12
    assert len(rows) == 20 and np.all(np.diff(rows) > 0)        # distinct scenes, ascending order
    assert np.array_equal(a, x0.numpy()[rows])                    # whole scenes, unchanged


def test_bench_rejects_bad_arguments(tmp_path):
    for argv in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
        assert p.returncode == 2 and "error:" in p.stderr, (argv, p.stderr)
