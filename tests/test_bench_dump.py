"""bench.py --dump-outputs writer (host logic): one .npy per output, float32 / float64, a fixed seeded sample above the size cap."""
import os
import numpy as np

import bench


def _outputs(n, rng):
    return {"obs": rng.standard_normal((n, 34)).astype(np.float32), "gc": rng.standard_normal((n, 19)).astype(np.float32),
            "gv": rng.standard_normal((n, 18)), "obs_e2e": rng.standard_normal((n, 34)).astype(np.float32)}


def test_writes_every_output_in_full_below_the_cap(tmp_path):
    arrays = _outputs(256, np.random.default_rng(1))
    bench.write_outputs(str(tmp_path), arrays)
    assert sorted(os.listdir(tmp_path)) == ["gc.npy", "gv.npy", "obs.npy", "obs_e2e.npy"]
    for k, a in arrays.items():
        b = np.load(tmp_path / (k + ".npy"))
        assert b.dtype == a.dtype and np.array_equal(a, b)


def test_samples_the_same_rows_of_every_output_above_the_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 60_000)
    arrays = _outputs(1000, np.random.default_rng(2))
    bench.write_outputs(str(tmp_path / "a"), arrays)
    bench.write_outputs(str(tmp_path / "b"), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["env_index.npy", "gc.npy", "gv.npy", "obs.npy", "obs_e2e.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 60_000
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert idx.dtype == np.float64 and 0 < len(idx) < 1000 and (np.diff(idx) > 0).all()
    for k, a in arrays.items():
        assert np.array_equal(np.load(tmp_path / "a" / (k + ".npy")), a[idx.astype(int)])
    for f in files:                                                         # the sample is fixed
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
