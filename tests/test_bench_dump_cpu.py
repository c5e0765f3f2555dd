"""bench.py argument checks, and --dump-outputs on host tensors: which arrays land in DIR, their dtypes, and that they are
the seeded sample and the per-grid sums of the grid handed in."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(monkeypatch):
    monkeypatch.syspath_prepend(ROOT)
    import bench

    return bench


@pytest.mark.parametrize("argv, ok", [(["--steps", "0"], False), (["--dump-outputs", "d", "--impl", "reference"], False),
                                      (["--steps", "1", "--dump-outputs", "d"], True)])
def test_parse_checks(monkeypatch, argv, ok):
    bench = _bench(monkeypatch)
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    if ok:
        a = bench.parse()
        assert a.steps == 1 and a.dump_outputs == "d"
    else:
        with pytest.raises(SystemExit):
            bench.parse()


def test_dump_outputs(tmp_path, monkeypatch):
    bench = _bench(monkeypatch)
    from moleculekit_b200 import workloads
    from moleculekit_b200.tools import voxeldescriptors as vd

    w = workloads.protein_pockets(B=3, n_atoms=200, box=16.0, radius=6.0, seed=4)
    batch = vd.VoxelBatch(w["coords"], w["sigmas"], boxsize=w["boxsize"], centers=w["centers"], voxelsize=w["voxelsize"])
    grid = torch.from_numpy(np.random.default_rng(1).random((batch.total_voxels, batch.C), dtype=np.float32))
    monkeypatch.setattr(bench, "DUMP_ROWS", 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), batch, grid)
    assert sorted(os.listdir(tmp_path / "a")) == ["occupancy_sample.npy", "occupancy_sum.npy"]
    for name in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)), name
    sample, sums = np.load(tmp_path / "a" / "occupancy_sample.npy"), np.load(tmp_path / "a" / "occupancy_sum.npy")
    rows = np.sort(np.random.default_rng(0).choice(batch.total_voxels, size=1000, replace=False))
    assert sample.dtype == np.float32 and np.array_equal(sample, grid.numpy()[rows])
    want = np.stack([g.astype(np.float64).sum(axis=0) for g in batch.split(grid.numpy())])
    assert sums.dtype == np.float64 and sums.shape == (3, batch.C) and np.allclose(sums, want, rtol=1e-12)
