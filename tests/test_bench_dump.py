"""bench.py --dump-outputs: the files it writes and the size cap (CPU only)."""
import numpy as np

import bench


def test_dump_outputs_writes_every_array_in_full(tmp_path):
    arrays = {"loss": np.array([1.5], np.float32), "grad.w": np.arange(12, dtype=np.float32).reshape(3, 4)}
    bench.dump_outputs(str(tmp_path / "out"), arrays)
    for name, a in arrays.items():
        got = np.load(tmp_path / "out" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, a)


def test_dump_outputs_over_the_cap_keeps_the_same_entries_every_run(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    rng = np.random.default_rng(0)
    arrays = {"a": rng.standard_normal(1000, dtype=np.float32), "b": rng.standard_normal((50, 40), dtype=np.float32)}
    bench.dump_outputs(str(tmp_path / "1"), arrays)
    bench.dump_outputs(str(tmp_path / "2"), arrays)
    total = 0
    for name, a in arrays.items():
        got = np.load(tmp_path / "1" / f"{name}.npy")
        total += got.nbytes
        assert 0 < got.size < a.size and np.isin(got, a).all()
        assert np.array_equal(got, np.load(tmp_path / "2" / f"{name}.npy"))
    assert total <= 4000
