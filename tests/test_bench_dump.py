"""CPU: what bench.py --dump-outputs writes."""
import numpy as np

import bench


def test_dump_outputs_keeps_every_pair_below_the_cap(tmp_path):
    mean, cov = np.arange(40, dtype=np.float32).reshape(5, 8), np.ones((5, 8, 8), np.float32)
    bench.dump_outputs(str(tmp_path / "out"), {"mean": mean, "cov": cov})
    assert np.array_equal(np.load(tmp_path / "out" / "mean.npy"), mean)
    assert np.array_equal(np.load(tmp_path / "out" / "cov.npy"), cov)


def test_dump_outputs_samples_the_same_pairs_of_every_array_above_the_cap(tmp_path, monkeypatch):
    n, per_pair = 1000, 72 * 4
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * per_pair)
    ids = np.arange(n, dtype=np.float32)
    arrays = {"mean": np.repeat(ids[:, None], 8, 1), "cov": np.repeat(ids[:, None], 64, 1).reshape(n, 8, 8)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    m, c = np.load(tmp_path / "a" / "mean.npy"), np.load(tmp_path / "a" / "cov.npy")
    assert m.shape == (100, 8) and c.shape == (100, 8, 8)
    assert np.array_equal(m[:, 0], c[:, 0, 0]) and np.all(np.diff(m[:, 0]) > 0)      # same pairs, in pair order
    assert np.array_equal(m, np.load(tmp_path / "b" / "mean.npy"))                   # the same sample on every run
