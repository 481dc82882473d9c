"""bench.py --dump-outputs on the host: what it writes, and that two runs on the same arrays write the same files."""
import os

import numpy as np
import pytest

import bench


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones_at_fixed_positions(tmp_path):
    n = 7 * (bench.DUMP_SAMPLE // 7 + 600)
    big = np.arange(n, dtype=np.float32).reshape((n // 7, 7), order="F")   # value = column-major position
    small = np.random.RandomState(0).standard_normal((3, 5)).astype(np.float32)
    arrays = {"big": big, "small": small, "loss": np.float64(-1.25)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "loss.npy", "small.npy"]
    s = np.load(tmp_path / "a" / "big.npy")
    assert s.dtype == np.float32 and s.shape == (bench.DUMP_SAMPLE,)
    assert (np.diff(s) > 0).all() and s[0] >= 0 and s[-1] < n                # distinct positions, in column-major order
    assert np.array_equal(s, np.load(tmp_path / "b" / "big.npy"))            # the same positions every run
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)
    loss = np.load(tmp_path / "a" / "loss.npy")
    assert loss.dtype == np.float64 and loss == -1.25


def test_dump_outputs_refuses_more_than_the_budget_and_non_float_arrays(tmp_path):
    x = np.zeros(bench.DUMP_SAMPLE, np.float64)
    n_fit = bench.DUMP_BUDGET // x.nbytes
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path / "over"), {f"x{i}": x for i in range(n_fit + 1)})
    assert not os.path.exists(tmp_path / "over")                              # nothing written
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path / "ints"), {"ids": np.arange(4)})
