"""CPU: bench.py --dump-outputs writes the solved field (whole, or a sample at seeded indices) and the solve statistics
that are not times, as float32 / float64 .npy files."""
import os

import numpy as np

import bench


def _dump(tmp_path, name, n, world=1, rank=0):
    import torch
    field = torch.arange(n, dtype=torch.float32) * 0.5
    stats = {"iterations": 400, "relative_residual": 1e-3, "converged": 0, "setup_ms": 1.5, "solve_ms": 2.5}
    out = str(tmp_path / name)
    bench.dump_outputs(out, field, stats, rank, world)
    return out, {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_small_field_is_written_whole(tmp_path):
    _, got = _dump(tmp_path, "a", 1000)
    assert sorted(got) == ["converged", "field", "iterations", "relative_residual"]
    assert got["field"].dtype == np.float32 and np.array_equal(got["field"], np.arange(1000, dtype=np.float32) * 0.5)
    assert got["iterations"].dtype == np.float64 and got["iterations"] == 400


def test_large_field_is_sampled_at_seeded_indices(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_FIELD_VALUES", 64)
    _, a = _dump(tmp_path, "a", 10_000)
    _, b = _dump(tmp_path, "b", 10_000)
    idx = a["field_index"]
    assert idx.dtype == np.float64 and idx.shape == (64,) and len(np.unique(idx)) == 64
    assert np.array_equal(idx, b["field_index"])
    assert np.array_equal(a["field"], (idx * 0.5).astype(np.float32))
    _, r1 = _dump(tmp_path, "c", 10_000, world=2, rank=1)
    assert r1["field_rank1"].shape == (32,) and "iterations_rank1" in r1


def test_default_sample_stays_under_64_mb(tmp_path):
    """A field just over the default sample size, on one rank and on two: what lands on disk is at most 64 MB."""
    for world in (1, 2):
        for rank in range(world):
            out, got = _dump(tmp_path, f"w{world}", bench.DUMP_FIELD_VALUES + 1, world, rank)
        assert sum(k.startswith("field_index") for k in got) == world
        total = sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out))
        assert total <= 64 << 20


def test_host_field_of_the_reference_arm(tmp_path):
    field = np.arange(5000, dtype=np.float32)
    bench.dump_outputs(str(tmp_path), field, {"iterations": 20, "relative_residual": 0.5}, 0, 1)
    assert np.array_equal(np.load(tmp_path / "field.npy"), field)
    assert np.load(tmp_path / "iterations.npy") == 20
