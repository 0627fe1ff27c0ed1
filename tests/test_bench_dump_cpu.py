"""bench.py --dump-outputs: what it writes and the fixed sample it falls back to past its size limit."""
import numpy as np
import torch

import bench


def test_dump_outputs_writes_float32_npy(tmp_path):
    out = torch.randn(2, 4, 1, 8, dtype=torch.bfloat16)
    bench.dump_outputs(str(tmp_path / "d"), {"out": out})
    a = np.load(tmp_path / "d" / "out.npy")
    assert a.dtype == np.float32 and a.shape == (2, 4, 1, 8)
    assert np.array_equal(a, out.float().numpy())


def test_dump_outputs_samples_large_results_the_same_way_every_run(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4 * 1000)
    x = torch.randn(3000)
    y = torch.randn(1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"x": x, "y": y})
    xa, ya = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "a" / "y.npy")
    assert xa.size + ya.size <= 1000 and xa.size == 750 and ya.size == 250
    assert np.array_equal(xa, np.load(tmp_path / "b" / "x.npy")) and np.array_equal(ya, np.load(tmp_path / "b" / "y.npy"))
    assert np.isin(xa, x.numpy()).all()
