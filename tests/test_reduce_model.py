"""The numpy model of the accumulate modes (tests/reduce_model.py) against the oracle, on clouds whose channel sums stay
below 2^24 (where an exact integer sum and CentroidPoint's float fold agree).  The GPU edge tests compare engine 2 with
this model where the oracle does not apply, so the model itself is pinned here.  CPU only."""
import numpy as np
import pytest

import oracle_binding as ob
import reduce_model as rm
from online_3d_reconstruction_b200 import abi


def _cloud(seed, n, span, heavy):
    rng = np.random.default_rng(seed)
    pts = np.zeros(n, dtype=abi.POINT)
    pts["x"] = rng.uniform(-span, span, n).astype(np.float32)
    pts["y"] = rng.uniform(-span / 2, span, n).astype(np.float32)
    pts["z"] = rng.uniform(-600.0, 900.0, n).astype(np.float32)   # several z cells of the 1000-high combined grid
    pts["rgb"] = rng.integers(0, 1 << 24, n, dtype=np.uint32)
    # one heavy cell with non-dyadic coordinates: the fold order changes bits there
    h = rng.choice(n, heavy, replace=False)
    pts["x"][h] = np.float32(0.0123) + rng.uniform(0, 0.03, heavy).astype(np.float32)
    pts["y"][h] = np.float32(-0.0377) + rng.uniform(0, 0.03, heavy).astype(np.float32)
    pts["z"][h] = np.float32(-499.9) + rng.uniform(0, 0.3, heavy).astype(np.float32)
    return pts


@pytest.mark.parametrize("seed,v,min_points", [(1, 0.05, 1), (2, 0.05, 3), (3, 0.25, 0), (4, 1.0, 2)])
def test_accumulate_model_matches_oracle(seed, v, min_points):
    pts = _cloud(seed, 20000, 3.0, 5000)
    p = abi.make_params(voxel_size=v, min_points_per_voxel=min_points)
    exp = ob.downsample_pt_cloud(p, pts, True)
    got, keys, counts = rm.accumulate_downsample(pts, v, min_points)
    assert got.shape == exp.shape
    assert np.array_equal(got.view(np.uint32), exp.view(np.uint32))
    assert np.all(np.diff(keys.astype(np.uint64)) > 0)
    assert counts.max() >= 5000 and counts.sum() <= len(pts)


def test_bright_cell_channel_cycle_separates_the_two_colour_sums():
    """150 000 points of one cell whose channel cycles 255, 253, 254: the float fold gives 253, the exact sum 254.  The
    GPU tests that use this cell rely on the two differing."""
    vals = np.tile(np.array([255, 253, 254], dtype=np.uint32), 50000)
    assert rm.float_fold_channel(vals) == 253
    assert rm.uint_sum_channel(vals) == 254


@pytest.mark.parametrize("seed,v", [(5, 0.05), (6, 0.25)])
def test_cell_sums_match_oracle(seed, v):
    """cell_sums (the exact per-cell sums the GPU tests compare exportCells() with) against the oracle's combined VoxelGrid:
    same cells in key order, and sums / n equal to its centroids (colours exact, coordinates within float rounding)."""
    pts = _cloud(seed, 20000, 3.0, 3000)
    p = abi.make_params(voxel_size=v, min_points_per_voxel=1)
    exp = ob.downsample_pt_cloud(p, pts, True)
    s = rm.cell_sums(pts, v)
    _, keys, counts = rm.accumulate_downsample(pts, v)
    assert np.array_equal(s["key"], keys) and np.array_equal(s["n"], counts) and s["n"].sum() == len(pts)
    assert len(s) == len(exp) and s["n"].max() >= 3000
    n = s["n"].astype(np.float32)
    rgb = [(s[f].astype(np.float32) / n).astype(np.uint32) for f in ("sr", "sg", "sb")]
    assert np.array_equal((rgb[0] << np.uint32(16)) | (rgb[1] << np.uint32(8)) | rgb[2], exp["rgb"])
    for f, a, sh in (("sx", "ax", 0.0), ("sy", "ay", 0.0), ("sz", "az", 500.0)):
        c = s[f] / s["n"]
        e = exp[f[1]].astype(np.float64) + sh
        assert np.all(np.abs(c - e) <= 1e-5 * s[a] / s["n"])   # the oracle folds in float32
