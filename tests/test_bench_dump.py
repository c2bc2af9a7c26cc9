"""bench.py --dump-outputs (host logic, no GPU): the last step's logits as float32 .npy, a fixed row sample above the size cap."""
import numpy as np
import torch

import bench


def test_dump_outputs_writes_the_logits_unchanged(tmp_path):
    x = torch.randn(8, 1000)
    path = bench.dump_outputs(str(tmp_path / "out"), x, 0, 1)
    assert path == str(tmp_path / "out" / "logits.npy")
    a = np.load(path)
    assert a.dtype == np.float32 and np.array_equal(a, x.numpy())


def test_dump_outputs_keeps_a_fixed_stride_of_rows_under_the_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 80_000)
    x = torch.randn(25, 1000)                                  # 100 kB: every second row fits 80 kB
    a = np.load(bench.dump_outputs(str(tmp_path), x, 0, 1))
    assert np.array_equal(a, x.numpy()[::2])
    # two ranks share the cap: 40 kB each, every third row
    b = np.load(bench.dump_outputs(str(tmp_path), x.bfloat16(), 1, 2))
    assert (tmp_path / "logits_rank1.npy").exists() and b.dtype == np.float32
    assert np.array_equal(b, x.bfloat16().float().numpy()[::3]) and b.nbytes <= 40_000
