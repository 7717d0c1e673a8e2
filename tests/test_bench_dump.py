"""bench.py --dump-outputs (host side): float32 arrays, within the size budget, the same sampled rows on every run."""
import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_is_float32_bounded_and_repeatable(tmp_path, monkeypatch):
    small = torch.randn(6, 4, 2, 2, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "small"), {"latents": small})
    got = np.load(tmp_path / "small" / "latents.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.float().numpy())

    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4096 + 10 * 64)        # header room + ten rows of 16 floats
    big = torch.randn(100, 4, 2, 2)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"latents": big})
    a, b = (np.load(tmp_path / run / "latents.npy") for run in ("a", "b"))
    assert a.shape == (10, 4, 2, 2) and np.array_equal(a, b)
    rows = [int(np.flatnonzero((big.numpy() == r).all(axis=(1, 2, 3)))[0]) for r in a]
    assert rows == sorted(set(rows))                                      # distinct rows of the output, in order

    with pytest.raises(ValueError, match="exceeds"):                       # a row above the budget: no empty sample
        bench.dump_outputs(str(tmp_path / "wide"), {"latents": torch.randn(3, 4096)})
