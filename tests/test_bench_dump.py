"""CPU: bench.py --dump-outputs keeps to its size budget with the same fixed sample of envs in every per-env array."""
import os

import numpy as np
import torch

import bench


def _read(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_samples_the_same_envs_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    n = 1000
    arrays = {"h": torch.arange(n * 40, dtype=torch.float32).view(n, 40), "done": torch.arange(n) % 2 == 0,
              "idx": np.arange(n, dtype=np.float64), "losses": torch.tensor([1.0, 2.0, 3.0])}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, n)
    a, b = _read(tmp_path / "a"), _read(tmp_path / "b")
    assert sorted(a) == ["done", "h", "idx", "losses"]
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= 100_000
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert a["h"].dtype == np.float32 and a["done"].dtype == np.float32 and a["idx"].dtype == np.float64
    rows = a["idx"].astype(np.int64)
    assert 0 < len(rows) < n and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["h"], arrays["h"].numpy()[rows]) and np.array_equal(a["done"], (rows % 2 == 0).astype(np.float32))
    assert np.array_equal(a["losses"], [1.0, 2.0, 3.0])


def test_dump_outputs_writes_everything_below_the_budget(tmp_path):
    n = 16
    arrays = {"h": torch.randn(n, 6, 256), "value": torch.randn(n, 1)}
    bench.dump_outputs(str(tmp_path), arrays, n)
    got = _read(tmp_path)
    assert all(np.array_equal(got[k], arrays[k].numpy()) for k in arrays)
