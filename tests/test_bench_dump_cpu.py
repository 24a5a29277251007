"""CPU: what `bench.py --dump-outputs` writes (bench.dump_outputs) -- whole arrays in float64 under the size cap, past
it the same seeded sample of every array on every run, within the cap."""
import os

import numpy as np

import bench


def test_dump_outputs_writes_whole_arrays_under_the_cap(tmp_path):
    x, z = np.arange(10, dtype=np.float32), -np.arange(20.0)
    bench.dump_outputs(tmp_path, {"x": x, "z": z})
    assert sorted(os.listdir(tmp_path)) == ["x.npy", "z.npy"]
    ex, ez = np.load(tmp_path / "x.npy"), np.load(tmp_path / "z.npy")
    assert ex.dtype == ez.dtype == np.float64
    assert np.array_equal(ex, x) and np.array_equal(ez, z)


def test_dump_outputs_samples_past_the_cap_within_it_and_reproducibly(tmp_path):
    # entry i of every array holds i, so a written array is the list of the indices it kept
    arrays = {"x": np.arange(100_000.0), "z": np.arange(150_000.0), "s": np.arange(150_000.0)}
    total, cap = 8 * 400_000, 1_000_000
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, arrays, cap=cap)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= cap
    for name, full in arrays.items():
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, b)           # the same sample on every run
        assert a.size == full.size * (cap - 4096 * len(arrays)) // total  # each array keeps its share of the cap
        assert np.all(np.diff(a) > 0) and a[0] >= 0 and a[-1] < full.size  # distinct indices, in order
        assert a[-1] > a.size                                            # spread over the array, not a prefix
