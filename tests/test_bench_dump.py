"""CPU: what bench.py --dump-outputs writes -- float32 arrays, within its size bound, the same elements on every run."""

import numpy as np
import torch

import bench


def test_dump_outputs_writes_float32(tmp_path):
    t = torch.randn(3, 5, dtype=torch.float16)
    (p,) = bench.dump_outputs(str(tmp_path), {"logits": t}, 0, 1)
    assert p == str(tmp_path / "logits.npy")
    a = np.load(p)
    assert a.dtype == np.float32 and np.array_equal(a, t.float().numpy())


def test_dump_outputs_samples_large_arrays(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1024)
    t = torch.arange(10000, dtype=torch.float32).reshape(100, 100)
    paths = [bench.dump_outputs(str(tmp_path), {"logits": t}, r, 2)[0] for r in (0, 1)]
    assert paths == [str(tmp_path / "logits.rank0.npy"), str(tmp_path / "logits.rank1.npy")]
    a, b = (np.load(p) for p in paths)
    assert a.nbytes + b.nbytes <= 1024
    assert np.array_equal(a, b)  # the same sample on every call
    assert (np.diff(a) > 0).all() and a[0] >= 0 and a[-1] < 10000  # distinct elements of the output, in order
