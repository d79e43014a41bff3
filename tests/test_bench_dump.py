"""bench.py --dump-outputs: float32 / float64 .npy files within the byte budget, large outputs as a fixed sample of their rows,
the same files from run to run."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_fits_the_budget_and_is_repeatable(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 40_000)
    g = torch.Generator().manual_seed(3)
    arrays = {"x": torch.randn((4, 50, 1), generator=g), "H": torch.randn((4, 90, 32), generator=g),
              "pri": torch.rand((10, 4), generator=g, dtype=torch.float64), "metrics": None}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    a, b = tmp_path / "a", tmp_path / "b"
    files = sorted(os.listdir(a))
    assert files == ["H.npy", "H_rows.npy", "pri.npy", "x.npy"]
    assert sum(os.path.getsize(a / f) for f in files) <= 40_000
    for f in files:
        assert np.load(a / f).dtype in (np.float32, np.float64)
        assert np.array_equal(np.load(a / f), np.load(b / f)), f
    assert np.load(a / "pri.npy").dtype == np.float64
    assert np.array_equal(np.load(a / "x.npy"), arrays["x"].numpy())
    rows = np.load(a / "H_rows.npy").astype(np.int64)
    assert 0 < len(rows) < 4 * 90 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(a / "H.npy"), arrays["H"].reshape(-1, 32).numpy()[rows])
