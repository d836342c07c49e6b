"""bench.py --dump-outputs: the output is written as float32, whole when it is small, as a fixed sample of token rows
(at most 64 MB with the .npy header) when it is large, and identically from run to run."""
import numpy as np
import torch

import bench


def test_small_output_is_written_whole(tmp_path):
    out = torch.randn(1, 300, 2, 128).to(torch.bfloat16)
    bench.dump_outputs(str(tmp_path), out)
    got = np.load(tmp_path / "output.npy")
    assert got.dtype == np.float32 and np.array_equal(got, out[0].float().numpy())
    assert bench.DUMP_BYTES + 4096 <= 64 * 10 ** 6


def test_large_output_is_sampled_by_row_with_a_fixed_seed(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * 2 * 128 * 4)
    out = torch.randn(1, 1000, 2, 128)
    out[0, :, 0, 0] = torch.arange(1000, dtype=torch.float32)      # each row carries its index
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    got = np.load(tmp_path / "a" / "output.npy")
    assert got.dtype == np.float32 and got.shape == (100, 2, 128)
    rows = got[:, 0, 0].astype(np.int64)
    assert np.all(np.diff(rows) > 0) and np.array_equal(got, out[0].numpy()[rows])
    assert np.array_equal(got, np.load(tmp_path / "b" / "output.npy"))
