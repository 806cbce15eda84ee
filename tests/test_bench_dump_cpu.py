"""CPU: bench.py --dump-outputs writes what a search returned as .npy files: ids as float64, values as float32, and a fixed,
seeded sample of query rows (with their row numbers) once the arrays would exceed the size bound."""
import os

import numpy as np
import torch

import bench


def _outputs(rows, k=10):
    g = torch.Generator().manual_seed(0)
    return {"distances": torch.rand((rows, k), generator=g),
            "neighbors": torch.arange(rows * k, dtype=torch.int64).reshape(rows, k) + (1 << 40)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dtypes_and_values_below_the_bound(tmp_path):
    out = _outputs(1000)
    cagra_ids = torch.arange(10_000, dtype=torch.int32).reshape(1000, 10).to(torch.uint32)
    bench.dump_outputs({**out, "graph_ids": cagra_ids}, str(tmp_path))
    got = _load(tmp_path)
    assert sorted(got) == ["distances", "graph_ids", "neighbors"]
    assert got["distances"].dtype == np.float32 and got["neighbors"].dtype == np.float64 and got["graph_ids"].dtype == np.float64
    np.testing.assert_array_equal(got["distances"], out["distances"].numpy())
    np.testing.assert_array_equal(got["neighbors"], out["neighbors"].numpy().astype(np.float64))  # exact below 2**53
    np.testing.assert_array_equal(got["graph_ids"], np.arange(10_000).reshape(1000, 10))


def test_large_outputs_keep_the_same_seeded_row_sample_within_64_mb(tmp_path):
    out = _outputs(1_000_000)  # 40 MB of float32 distances + 80 MB of float64 ids
    for run in ("a", "b"):
        bench.dump_outputs(out, str(tmp_path / run))
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64_000_000
    rows = a["rows"].astype(np.int64)
    assert len(rows) > 0 and (np.diff(rows) > 0).all() and rows[-1] < 1_000_000
    for name in a:
        np.testing.assert_array_equal(a[name], b[name])
    np.testing.assert_array_equal(a["distances"], out["distances"].numpy()[rows])
    np.testing.assert_array_equal(a["neighbors"], out["neighbors"].numpy()[rows].astype(np.float64))
