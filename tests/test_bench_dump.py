"""CPU tests of `bench.py --dump-outputs`: file names, dtypes, the size budget and the seeded row sample."""
import os

import numpy as np
import torch

import bench


def test_dump_writes_every_output_as_float_npy(tmp_path):
    logits = torch.randn(2, 8, 1)
    bench.dump_outputs(str(tmp_path), {"logits": logits, "half": logits.half(), "wide": logits.double(), "AUC": 0.75,
                                       "classwise": [[0.5, 0.25], [1.0, 0.125]]})
    assert sorted(os.listdir(tmp_path)) == ["AUC.npy", "classwise.npy", "half.npy", "logits.npy", "wide.npy"]
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert got["logits"].dtype == np.float32 and np.array_equal(got["logits"], logits.numpy())
    assert got["half"].dtype == np.float32 and np.array_equal(got["half"], logits.half().float().numpy())
    assert got["wide"].dtype == np.float64 and np.array_equal(got["wide"], logits.double().numpy())
    assert got["AUC"].dtype == np.float64 and got["AUC"].shape == () and float(got["AUC"]) == 0.75
    assert got["classwise"].shape == (2, 2) and got["classwise"][1, 1] == 0.125


def test_dump_samples_large_outputs_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    rows = torch.arange(64 * 256, dtype=torch.float32)
    wide = rows[:, None].repeat(1, 128).reshape(64, 256, 128)          # every row holds its own index
    outputs = {"wide": wide, "scores": rows, "logits": rows.reshape(64, 256, 1), "long": torch.arange(1 << 20) * 0.5}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outputs)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= (1 << 20) + 4 * 128                                 # payload within the budget, plus .npy headers
    for name in outputs:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert np.array_equal(a, b)                                     # the same sample on every run
    w = np.load(tmp_path / "a" / "wide.npy")
    assert w.shape[1] == 128 and 0 < w.shape[0] < 64 * 256
    assert np.all(w == w[:, :1]) and np.all(np.diff(w[:, 0]) > 0)       # whole rows, ascending, no repeats
    long = np.load(tmp_path / "a" / "long.npy")
    assert long.dtype == np.float32 and long.ndim == 1 and 0 < long.size < 1 << 20 and np.all(np.diff(long) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "scores.npy"), rows.numpy())          # within its share: whole
    assert np.array_equal(np.load(tmp_path / "a" / "logits.npy"), rows.reshape(64, 256, 1).numpy())
