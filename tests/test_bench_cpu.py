"""CPU: bench.py's argument checks and the writer behind --dump-outputs (float32 .npy files, whole below the
size cap, the same seeded sample of every array above it)."""
import sys

import numpy as np
import pytest

import bench


def parse(monkeypatch, *argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    return bench.parse()


def test_steps_sets_the_timed_steps_and_must_be_positive(monkeypatch):
    assert parse(monkeypatch, "--steps", "7", "--warmup", "0").steps == 7
    for bad in ("0", "-3"):
        with pytest.raises(SystemExit):
            parse(monkeypatch, "--steps", bad)


def test_dump_outputs_needs_the_gpu_implementation(monkeypatch):
    assert parse(monkeypatch, "--dump-outputs", "out").dump_outputs == "out"
    with pytest.raises(SystemExit):
        parse(monkeypatch, "--impl", "reference", "--dump-outputs", "out")


def test_dump_writes_arrays_below_the_cap_whole_in_float32(tmp_path):
    rng = np.random.default_rng(0)
    arrays = {"metrics": rng.standard_normal(8).astype(np.float32), "actor.0.weight": rng.standard_normal((16, 5)),
              "actor.0.bias": rng.standard_normal(16).astype(np.float32)}
    bench.dump_outputs(str(tmp_path / "out"), arrays)
    assert sorted(p.name for p in (tmp_path / "out").iterdir()) == sorted(f"{k}.npy" for k in arrays)
    for name, v in arrays.items():
        got = np.load(tmp_path / "out" / f"{name}.npy")
        assert got.dtype == np.float32 and got.shape == v.shape
        np.testing.assert_array_equal(got, v.astype(np.float32))


def test_dump_above_the_cap_writes_the_same_sample_every_time(tmp_path):
    rng = np.random.default_rng(1)
    arrays = {"a": rng.standard_normal((300, 100)), "b": rng.standard_normal(1000).astype(np.float32)}
    budget = 4 * 2000
    for d in ("x", "y"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=budget)
    total = 0
    for name, v in arrays.items():
        x, y = np.load(tmp_path / "x" / f"{name}.npy"), np.load(tmp_path / "y" / f"{name}.npy")
        assert x.dtype == np.float32 and x.size < v.size
        np.testing.assert_array_equal(x, y)
        assert np.isin(x, v.astype(np.float32).ravel()).all()
        total += x.nbytes
    assert 0.9 * budget < total <= budget
