"""CPU: bench.py --dump-outputs writes each output as float32 (float64 stays float64), 64 MB at most in all, and samples a
large output at the same positions on every run."""
import os

import numpy as np


def test_dump_outputs_dtype_budget_and_fixed_sample(tmp_path):
    import torch
    import bench
    depth = torch.arange(12, dtype=torch.int32).reshape(3, 4).to(torch.uint16)
    big = torch.randint(0, 256, (10, 1000, 1000, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(0))
    exact = torch.linspace(0, 1, 7, dtype=torch.float64)
    outs, names = (depth, big, exact), ("depth", "big", "exact")
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), names, outs)
    files = {n: str(tmp_path / "a" / f"{n}.npy") for n in names}
    assert sum(os.path.getsize(f) for f in files.values()) <= 64 << 20
    got = {n: np.load(f) for n, f in files.items()}
    assert got["depth"].dtype == np.float32 and np.array_equal(got["depth"], depth.numpy().astype(np.float32))
    assert got["exact"].dtype == np.float64 and np.array_equal(got["exact"], exact.numpy())
    assert got["big"].dtype == np.float32 and got["big"].ndim == 1 and 0 < got["big"].size < big.numel()
    assert np.isin(got["big"], np.arange(256)).all()
    for n in names:
        assert np.array_equal(got[n], np.load(str(tmp_path / "b" / f"{n}.npy")))
