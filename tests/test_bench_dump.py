"""bench.py --dump-outputs: what the files hold (CPU only, no benchmark run)."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_writes_the_whole_result(tmp_path):
    D = torch.rand(7, 5)
    I = torch.randint(0, 1 << 40, (7, 5))
    bench.dump_outputs(str(tmp_path), D, I)
    d, i = np.load(tmp_path / "distances.npy"), np.load(tmp_path / "labels.npy")
    assert d.dtype == np.float32 and i.dtype == np.float64
    assert np.array_equal(d, D.numpy()) and np.array_equal(i.astype(np.int64), I.numpy())
    assert sorted(os.listdir(tmp_path)) == ["distances.npy", "labels.npy"]


def test_dump_outputs_samples_a_large_result(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1000)
    D = torch.rand(200, 10)
    I = torch.arange(2000).reshape(200, 10)
    bench.dump_outputs(str(tmp_path / "a"), D, I)
    bench.dump_outputs(str(tmp_path / "b"), D, I)
    rows = np.load(tmp_path / "a" / "query_rows.npy")
    assert rows.dtype == np.float64 and rows.size > 1
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 1000  # headers included
    assert np.array_equal(rows, np.load(tmp_path / "b" / "query_rows.npy"))  # the same sample every run
    r = rows.astype(np.int64)
    assert np.all(np.diff(r) > 0) and r[-1] < 200
    assert np.array_equal(np.load(tmp_path / "a" / "distances.npy"), D.numpy()[r])
    assert np.array_equal(np.load(tmp_path / "a" / "labels.npy"), I.numpy()[r].astype(np.float64))
