"""bench.py --dump-outputs: arrays are written whole in float32 / float64, or as the same seeded sample on every run
when they exceed the size budget."""
import numpy as np

import bench


def test_small_outputs_are_written_whole(tmp_path):
    bench.dump_outputs(str(tmp_path), {"params": np.arange(12, dtype=np.float32).reshape(3, 4),
                                       "adam_step": np.array([5, 6], dtype=np.int32)})
    params, step = np.load(tmp_path / "params.npy"), np.load(tmp_path / "adam_step.npy")
    assert params.dtype == np.float32 and np.array_equal(params, np.arange(12).reshape(3, 4))
    assert step.dtype == np.float64 and step.tolist() == [5.0, 6.0]


def test_large_outputs_are_sampled_the_same_way_on_every_run(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    arrays = {"value": np.random.default_rng(1).standard_normal(1000).astype(np.float32), "losses": np.arange(1000.0)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    total = 0
    for name, full in arrays.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == full.dtype and len(a) == 333 and np.array_equal(a, b) and np.isin(a, full).all()
        total += a.nbytes
    assert total <= 4000
    assert (np.diff(np.load(tmp_path / "a" / "losses.npy")) > 0).all()      # sampled elements keep their order
