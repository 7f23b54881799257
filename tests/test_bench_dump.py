"""bench.py --dump-outputs: dtypes, the size limit and the seeded instance sample (on CPU tensors)."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_writes_a_small_batch_whole(tmp_path):
    outs = dict(pilots=torch.rand(3, 4, 5, dtype=torch.float64), stats=torch.rand(3, 2), status=torch.tensor([0, 1, 0], dtype=torch.int32))
    bench.dump_outputs(str(tmp_path), outs)
    assert np.load(tmp_path / "instance.npy").tolist() == [0.0, 1.0, 2.0]
    for name, t in outs.items():
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == (np.float32 if t.dtype == torch.float32 else np.float64)
        np.testing.assert_array_equal(a, t.numpy())


def test_dump_outputs_samples_the_same_instances_within_the_limit(tmp_path, monkeypatch):
    per_instance = 8 + 6 * 8 + 8 + 4  # index, pilots, iters (as float64), stats
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 100 * per_instance)
    B = 1000
    outs = dict(pilots=torch.arange(B * 6, dtype=torch.float64).reshape(B, 2, 3), iters=torch.arange(B, dtype=torch.int32),
                stats=torch.arange(B, dtype=torch.float32))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outs)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["instance.npy", "iters.npy", "pilots.npy", "stats.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    idx = np.load(tmp_path / "a" / "instance.npy").astype(np.int64)
    assert len(idx) == 100 and np.all(np.diff(idx) > 0) and idx[-1] < B
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "pilots.npy"), outs["pilots"].numpy()[idx])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "iters.npy"), idx.astype(np.float64))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "stats.npy"), idx.astype(np.float32))
    for f in files:
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
