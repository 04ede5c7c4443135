"""bench.py's command line and its --dump-outputs writer (host logic; the timed path itself needs the GPU)."""
import sys

import numpy as np
import pytest
import torch

import bench


def test_steps_must_be_positive(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "5", "--dump-outputs", "out"])
    a = bench.parse()
    assert a.steps == 5 and a.dump_outputs == "out"


def test_dump_outputs_names_and_dtypes(tmp_path):
    arrays = {"logprob": torch.randn(1, 64), "gcn_feat": torch.randn(1, 64, 32).half(),
              "nll_acc": torch.tensor([-3.5, 64.0], dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path), arrays)
    for name, t in arrays.items():
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == (np.float64 if t.dtype == torch.float64 else np.float32), name
        np.testing.assert_array_equal(a, t.double().numpy())


def test_dump_outputs_samples_rows_past_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT", 64 * 4 + 100 * 32 * 4)
    feat = torch.randn(1, 1000, 32)
    arrays = {"logprob": torch.randn(1, 64), "gcn_feat": feat}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "logprob.npy"), arrays["logprob"].numpy())     # fits: whole
    got = np.load(tmp_path / "a" / "gcn_feat.npy")
    assert got.shape == (100, 32)
    np.testing.assert_array_equal(got, np.load(tmp_path / "b" / "gcn_feat.npy"))                          # a fixed sample
    rows = feat.reshape(-1, 32).numpy()
    idx = [int(np.flatnonzero((rows == r).all(1))[0]) for r in got]
    assert idx == sorted(set(idx))                                                                         # distinct, in order
