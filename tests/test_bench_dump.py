"""bench.py --dump-outputs: dtypes, the 64 MB cap and a row sample that is the same on every run."""
import numpy as np
import torch

import bench


def test_dump_outputs_keeps_dtypes_budget_and_rows(tmp_path):
    n = 16_000_000                     # float32 holds every row number below 2^24
    g = torch.Generator().manual_seed(1)
    outs = {"coeffs": torch.randn(32, dtype=torch.float64, generator=g), "status": torch.zeros(1, dtype=torch.int32),
            "pred": torch.arange(n, dtype=torch.float32), "valid": torch.ones(n, dtype=torch.uint8)}
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), outs)
    bench.dump_outputs(str(b), outs)
    assert sum(f.stat().st_size for f in a.iterdir()) <= 64 << 20
    got = {f.stem: np.load(f) for f in a.iterdir()}
    assert sorted(got) == ["coeffs", "pred", "status", "valid"]
    assert got["coeffs"].dtype == np.float64 and np.array_equal(got["coeffs"], outs["coeffs"].numpy())
    assert got["status"].dtype == got["pred"].dtype == got["valid"].dtype == np.float32
    rows = got["pred"].astype(np.int64)                      # pred[i] == i: the sample's row numbers
    assert 1_000_000 < len(rows) < n and np.all(np.diff(rows) > 0) and len(got["valid"]) == len(rows)
    for f in a.iterdir():
        assert np.array_equal(np.load(f), np.load(b / f.name))
