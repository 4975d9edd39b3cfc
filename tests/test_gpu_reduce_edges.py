"""Structural edges of the radix sort and the run reductions, against plain references.

The other GPU tests use clouds where no cell holds more than a few hundred items.  Here the cells are heavy enough to
cross reduce tiles (kTileV = 1024 items: the RunCarry hand-off, tiles with no run head of their own, engine 2's
continuation of a resident cell), the clouds sit at radix-tile edges (kRsTile = 4096 pairs: partial last tiles whose
real items share the padding's all-ones digit, 1-bit and 32-bit keys), on PCL's int32 index wrap and pass-through
threshold, on engine 2's 64-bit compact key and its +-2^20 cell limit, and at 2^30 items in one sorted segment.

References: the oracle (bit for bit: keys, counts, order, centroids, colours) wherever its semantics apply, else the
numpy model of the accumulate modes in reduce_model.py (itself checked against the oracle in test_reduce_model.py).
Inputs are shuffled with a seed, so the fold order inside a cell is input order, and heavy cells have non-dyadic
coordinates, so a wrong fold order changes bits.
"""
import time

import numpy as np
import pytest

import oracle_binding as ob
import reduce_model as rm
from online_3d_reconstruction_b200 import abi, lib
from online_3d_reconstruction_b200.pose import Pose

pytestmark = pytest.mark.gpu

F32 = np.float32
SMALL = dict(rows=120, cols=200)


def _eq(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    if not np.array_equal(a.view(np.uint32), b.view(np.uint32)):
        bad = np.nonzero(a.view(np.uint32).reshape(-1, 4) != b.view(np.uint32).reshape(-1, 4))[0]
        raise AssertionError(f"{len(np.unique(bad))} of {len(a)} records differ; first at {bad[0]}: {a[bad[0]]} vs {b[bad[0]]}")


def _points(x, y, z, rgb):
    p = np.zeros(len(x), dtype=abi.POINT)
    p["x"], p["y"], p["z"], p["rgb"] = np.asarray(x, F32), np.asarray(y, F32), np.asarray(z, F32), np.asarray(rgb, np.uint32)
    return p


def _rgb(rng, n, cmax=256):
    """n colours whose channels are each below cmax."""
    c = rng.integers(0, cmax, (3, n)).astype(np.uint32)
    return (c[0] << 16) | (c[1] << 8) | c[2]


def _in_cell(rng, lo, n, v):
    """n non-dyadic coordinates inside the cell [lo * v, (lo + 1) * v), away from its faces."""
    return (F32(lo) + rng.uniform(0.1, 0.9, n).astype(F32)) * F32(v)


def _retain(pts, v, min_points, pieces=1):
    p = abi.make_params(voxel_size=v, min_points_per_voxel=min_points, merge_mode=abi.MERGE_RETAIN, **SMALL)
    with Pose(p) as P:
        for part in np.array_split(pts, pieces):
            P.appendPoints(part)
        return P.downsamplePtCloud().copy()


def _oracle_retain(pts, v, min_points):
    return ob.downsample_pt_cloud(abi.make_params(voxel_size=v, min_points_per_voxel=min_points), pts, True)


def _probe(pts, leaf, min_points):
    with Pose(abi.make_params(**SMALL)) as P:
        return P.voxelGrid(pts, leaf, min_points)


def _check_probe(pts, leaf, min_points=0):
    g_pts, g_keys, g_cnt, g_pass = _probe(pts, leaf, min_points)
    e_pts, e_keys, e_cnt, e_pass = ob.voxel_grid(pts, leaf, min_points)
    assert g_pass == e_pass
    assert np.array_equal(g_keys, e_keys)
    assert np.array_equal(g_cnt, e_cnt)
    _eq(g_pts, e_pts)
    return g_pts, g_cnt, g_pass


# ----------------------------------------------------------------------------------------- heavy runs (engine 1)
V_HEAVY = 0.05
# cells in key (x) order.  Run starts (mod 1024): 0 (cells 0, 1, 7), 1 (2, 3), 2 (4), 1023 (the 3*1024+1 cell);
# the 150 000-point cell holds ~145 whole reduce tiles without a run head (H == 0) and 5000 ends mid-tile.
HEAVY_SIZES = [1024, 1, 1023, 1025, 2049, 1021, 3 * 1024 + 1, 5000] + [1] * 120 + [150000]


def _heavy_cloud(seed, rgb_max=256, light=3000):
    rng = np.random.default_rng(seed)
    parts = []
    for c, n in enumerate(HEAVY_SIZES):
        parts.append(_points(_in_cell(rng, c, n, V_HEAVY), _in_cell(rng, 3, n, V_HEAVY), _in_cell(rng, 1, n, V_HEAVY),
                             _rgb(rng, n, rgb_max)))
    # light cells after them: 1 to 4 points each
    lc = len(HEAVY_SIZES) + rng.integers(0, 4000, light)
    parts.append(_points(_in_cell(rng, 0, light, V_HEAVY) + lc.astype(F32) * F32(V_HEAVY), _in_cell(rng, 3, light, V_HEAVY),
                         _in_cell(rng, 1, light, V_HEAVY), _rgb(rng, light, rgb_max)))
    pts = np.concatenate(parts)
    return pts[rng.permutation(len(pts))]


@pytest.mark.parametrize("min_points", [1, 2])
def test_heavy_runs_retain_downsample(min_points):
    """RETAIN downsample through the tile hand-off of every heavy run: min_points 1 emits every run, 2 ranks the runs
    that pass the filter."""
    pts = _heavy_cloud(5)
    got = _retain(pts, V_HEAVY, min_points, pieces=3)
    _eq(got, _oracle_retain(pts, V_HEAVY, min_points))


@pytest.mark.parametrize("min_points", [0, 2, 1025])
def test_heavy_runs_voxel_grid_probe(min_points):
    pts = _heavy_cloud(6)
    _, cnt, _ = _check_probe(pts, (V_HEAVY, V_HEAVY, V_HEAVY), min_points)
    assert cnt.max() == 150000


def _bright_cloud(seed):
    """One 150 000-point cell whose red channel cycles 255, 253, 254 (float fold 253, exact sum 254), green cycles
    1, 2, 4 and blue is 200; its points keep their relative order but sit at seeded positions among light cells."""
    rng = np.random.default_rng(seed)
    n = 150000
    r = np.tile(np.array([255, 253, 254], np.uint32), n // 3)
    g = np.tile(np.array([1, 2, 4], np.uint32), n // 3)
    bright = _points(_in_cell(rng, 7, n, V_HEAVY), _in_cell(rng, 2, n, V_HEAVY), _in_cell(rng, 1, n, V_HEAVY),
                     (r << 16) | (g << 8) | np.uint32(200))
    m = 20000
    other = _points(_in_cell(rng, 0, m, V_HEAVY) + rng.integers(0, 40, m).astype(F32) * F32(V_HEAVY),
                    _in_cell(rng, 0, m, V_HEAVY) + (5 + rng.integers(0, 5, m)).astype(F32) * F32(V_HEAVY),   # y cells 5..9
                    _in_cell(rng, 1, m, V_HEAVY), rng.integers(0, 1 << 24, m))
    out = np.empty(n + m, dtype=abi.POINT)
    at = np.sort(rng.choice(n + m, n, replace=False))
    mask = np.zeros(n + m, dtype=bool)
    mask[at] = True
    out[mask] = bright
    out[~mask] = other[rng.permutation(m)]
    return out, r


def test_bright_cell_retain_colour_matches_pcl():
    """The RETAIN downsample folds colour channels as floats, as PCL's CentroidPoint does, with and without the
    min-points filter: min_points 1 and 2 give the oracle's record."""
    pts, r = _bright_cloud(7)
    assert rm.float_fold_channel(r) != rm.uint_sum_channel(r)   # the cell separates the two colour sums
    exp = _oracle_retain(pts, V_HEAVY, 1)
    a = _retain(pts, V_HEAVY, 1)
    b = _retain(pts, V_HEAVY, 2)
    _eq(a, exp)
    _eq(b, _oracle_retain(pts, V_HEAVY, 2))
    rec = a[(a["x"] > F32(7 * V_HEAVY)) & (a["x"] < F32(8 * V_HEAVY)) & (a["y"] > F32(2 * V_HEAVY)) & (a["y"] < F32(3 * V_HEAVY))]
    assert len(rec) == 1 and int(rec["rgb"][0]) >> 16 == rm.float_fold_channel(r)
    ib = np.nonzero((b["x"] == rec["x"][0]) & (b["y"] == rec["y"][0]))[0]
    assert len(ib) == 1 and b["rgb"][ib[0]] == rec["rgb"][0]


# ------------------------------------------------------------------------------------------------ radix edges
RADIX_SIZES = [4095, 4096, 4097, 3 * 4096 - 1, 3 * 4096 + 1, (1 << 20) + 3]


def _radix_cloud(n, dist, seed):
    rng = np.random.default_rng(seed)
    if dist == "distinct":         # every point its own cell
        cx = rng.permutation(n)
    elif dist == "one":            # one cell: every pass trivial, the reduction reads the points in place
        cx = np.full(n, 5)
    elif dist == "two":            # two cells: a 1-bit key
        cx = rng.integers(0, 2, n)
    else:                          # 16-bit key, mostly cells whose top digit is all ones (the padding's digit)
        cx = np.where(rng.random(n) < 0.9, rng.integers(0xff00, 0x10000, n), rng.integers(0, 0x10000, n))
        cx[:2] = (0, 0xffff)
        cx = cx[rng.permutation(n)]
    x = _in_cell(rng, 0, n, 1.0) + cx.astype(F32)
    return _points(x, _in_cell(rng, 0, n, 1.0), rng.uniform(0.1, 0.4, n), rng.integers(0, 1 << 24, n))


@pytest.mark.parametrize("dist", ["distinct", "one", "two", "top"])
@pytest.mark.parametrize("n", RADIX_SIZES)
def test_radix_edges(n, dist):
    pts = _radix_cloud(n, dist, n % 1000 + len(dist))
    _check_probe(pts, (1.0, 1.0, 1.0))
    _eq(_retain(pts, 1.0, 1), _oracle_retain(pts, 1.0, 1))


# -------------------------------------------------------------------------------------- grid guard (leaf 1)
def _guard_cloud(seed, lo, hi, zlo, zhi, n=50000):
    rng = np.random.default_rng(seed)
    corners = _points([lo[0], hi[0]], [lo[1], hi[1]], [zlo, zhi], [0x102030, 0x405060])
    body = _points(rng.uniform(lo[0], hi[0], n), rng.uniform(lo[1], hi[1], n), rng.uniform(zlo, zhi, n),
                   rng.integers(0, 1 << 24, n))
    return np.concatenate([corners, body])


@pytest.mark.parametrize("hi,passthrough", [((46339.9, 46340.9), False), ((46340.9, 46340.9), True)])
def test_guard_threshold(hi, passthrough):
    """d = 46340 * 46341 fits int32 (kept, 31 live key bits), d = 46341^2 does not (output = input)."""
    pts = _guard_cloud(9, (0.5, 0.5), hi, 0.2, 0.7)
    got, _, gpass = _check_probe(pts, (1.0, 1.0, 1.0))
    assert gpass == passthrough
    if passthrough:
        _eq(got, pts)


def _wrapped_index(pts):
    """PCL's relative leaf index of the wrap window's grid (min_b = 0, div_b = 46341, 46341, 2), wrapped to 32 bits."""
    i = np.floor(pts["x"].astype(F32)).astype(np.uint64)
    j = np.floor(pts["y"].astype(F32)).astype(np.uint64)
    k = np.floor(pts["z"].astype(F32)).astype(np.uint64)
    return (i + j * np.uint64(46341) + k * np.uint64(46341 * 46341)) & np.uint64(0xffffffff)


def test_guard_index_wrap_merges_like_pcl():
    """x, y in [0.5, 46340.4], z in [0.7, 1.2]: the guard's d = 46340^2 * 1 fits int32 but div_b = 46341^2 * 2 does not, so
    the 32-bit index wraps.  (37075.5 + a, 46340.2, 1.1) and (a + 0.5, 0.5, 0.8) then share index a: PCL merges them."""
    a = 1234
    pts = _guard_cloud(10, (0.5, 0.5), (46340.4, 46340.4), 0.7, 1.2)
    pair = _points([37075.5 + a, a + 0.5], [46340.2, 0.5], [1.1, 0.8], [0xff0000, 0x0000ff])
    rng = np.random.default_rng(11)
    pts = np.concatenate([pts, pair])
    pts = pts[rng.permutation(len(pts))]
    wi = _wrapped_index(pts)
    assert np.all(_wrapped_index(pair) == a)
    got, cnt, gpass = _check_probe(pts, (1.0, 1.0, 1.0))
    assert not gpass
    first = pts[np.nonzero(wi == a)[0][0]]   # the record of index a carries the key of its first point
    _, keys, _, _ = ob.voxel_grid(pts, (1.0, 1.0, 1.0))
    rec = np.nonzero(keys == ob.cell_key(first["x"], first["y"], first["z"], (1.0, 1.0, 1.0)))[0]
    assert len(rec) == 1 and cnt[rec[0]] == int(np.sum(wi == a)) >= 2   # ONE record holds the pair
    assert len(got) == len(np.unique(wi))


@pytest.mark.parametrize("leaf", [0.05, 0.01, 0.25])
def test_float_cell_boundaries(leaf):
    """Points at k * leaf computed in float32 and one ulp either side, negative coordinates and -0.0."""
    rng = np.random.default_rng(int(leaf * 1000))
    k = np.arange(-60, 61).astype(F32)
    b = k * F32(leaf)
    xs = np.concatenate([b, np.nextafter(b, F32(-np.inf)), np.nextafter(b, F32(np.inf)), [F32(-0.0), F32(0.0)]])
    x = np.repeat(xs, 3)
    y = rng.choice(xs, len(x))
    z = np.where(rng.random(len(x)) < 0.5, F32(-0.0), rng.choice(xs, len(x)))
    pts = _points(x, y, z, rng.integers(0, 1 << 24, len(x)))
    pts = pts[rng.permutation(len(pts))]
    _check_probe(pts, (leaf, leaf, leaf))
    _check_probe(pts, (leaf, leaf, leaf), 2)


# ----------------------------------------------------------------------------- engine 2 (ACCUMULATE, 3 appends)
def _acc(pts_parts, v, min_points, track=False):
    p = abi.make_params(voxel_size=v, min_points_per_voxel=min_points, merge_mode=abi.MERGE_ACCUMULATE, **SMALL)
    with Pose(p) as P:
        if track:
            P.trackCloudChanges(True)
        for part in pts_parts:
            P.appendPoints(part)
        out = P.downsamplePtCloud().copy()
        ch = P.cloudChanges() if track else None
    return out, ch


def _split_resident_first(pts, seed):
    """Three appends; the first two hold ~a third of each heavy cell, so the third append extends resident cells
    across reduce tiles (k_acc_reduce continues the resident sums over the carry chain)."""
    rng = np.random.default_rng(seed)
    cut = np.sort(rng.choice(np.arange(1, len(pts)), 2, replace=False))
    return np.split(pts, cut)


@pytest.mark.parametrize("min_points", [1, 3])
def test_heavy_cells_accumulate_against_oracle(min_points):
    pts = _heavy_cloud(12, rgb_max=100)   # every channel sum stays below 2^24: the exact sums equal PCL's float fold
    parts = _split_resident_first(pts, 13)
    got, _ = _acc(parts, V_HEAVY, min_points)
    _eq(got, _oracle_retain(pts, V_HEAVY, min_points))
    _eq(got, rm.accumulate_downsample(pts, V_HEAVY, min_points)[0])


def test_bright_cell_accumulate_keeps_uint32_sums():
    """The accumulate modes keep exact uint32 colour sums (DESIGN §2): past 2^24 they differ from PCL's float fold."""
    pts, r = _bright_cloud(14)
    got, _ = _acc(_split_resident_first(pts, 15), V_HEAVY, 1)
    exp = rm.accumulate_downsample(pts, V_HEAVY, 1)[0]
    _eq(got, exp)
    rec = got[(got["x"] > F32(7 * V_HEAVY)) & (got["x"] < F32(8 * V_HEAVY)) & (got["y"] > F32(2 * V_HEAVY)) &
              (got["y"] < F32(3 * V_HEAVY))]
    assert len(rec) == 1 and int(rec["rgb"][0]) >> 16 == rm.uint_sum_channel(r)


# ------------------------------------------------------------------------------------------------- wide keys
def test_wide_compact_key_equals_model_and_narrow_pieces():
    """voxel_size 0.05, x over 2^17 cells and y over 2^16 cells: 33 bits of cell extent, so one append sorts the 64-bit
    compact key; appended as two y halves (32 bits each) it takes the 32-bit key.  Both equal the numpy model, and each
    other bit for bit (each cell's points arrive in the same order either way).  The oracle does not apply: PCL's int32
    guard trips on this extent and the reference would return cloud_big verbatim (the accumulate modes do not emulate
    that guard on the combined grid)."""
    v = 0.05
    rng = np.random.default_rng(16)
    n = 400000
    ci = rng.integers(0, 1 << 17, n)
    cj = rng.integers(0, 1 << 16, n)
    ci[:2], cj[:2] = (0, (1 << 17) - 1), (0, (1 << 16) - 1)
    hot = rng.integers(0, 300, n // 4)   # heavy cells: ~330 points each
    ci[n // 2: n // 2 + len(hot)] = hot * 401 + 7
    cj[n // 2: n // 2 + len(hot)] = hot * 211 + 3
    pts = _points(_in_cell(rng, 0, n, v) + ci.astype(F32) * F32(v), _in_cell(rng, 0, n, v) + cj.astype(F32) * F32(v),
                  rng.uniform(-499.0, 400.0, n), rng.integers(0, 1 << 24, n))
    pts = pts[rng.permutation(n)]
    i, j, k = rm.cells(pts, v)
    assert i.max() - i.min() + 1 == 1 << 17 and j.max() - j.min() + 1 == 1 << 16 and k.min() == k.max()
    exp = rm.accumulate_downsample(pts, v, 1)[0]
    one, _ = _acc([pts], v, 1)
    _eq(one, exp)
    low = j < j.min() + (1 << 15)
    two, _ = _acc([pts[low], pts[~low]], v, 1)
    _eq(two, one)


def _cell_coord(c, v):
    """A float32 coordinate whose combined-grid cell (floor(x * (1/v))) is exactly c."""
    x = F32((c + 0.5) * v)
    assert int(np.floor(x * (F32(1) / F32(v)))) == c
    return x


def _z_of_cell(c):
    """A float32 z whose combined-grid z cell (floor((z + 500) * (1/1000))) is exactly c."""
    z = F32((c + 0.5) * 1000.0 - 500.0)
    assert int(np.floor((z + F32(500)) * (F32(1) / F32(1000)))) == c
    return z


def test_cell_limit_accepted_and_refused():
    """Cells +-(2^20 - 1) on each axis are accepted (key fields 1 and 2^21 - 1); a cell at +-2^20 on any axis, a NaN or an
    inf point returns O3R_ERR_INVALID and leaves the resident cloud as it was."""
    L = (1 << 20) - 1
    v = 1.0
    ext = []
    for sx in (-L, L):
        for sy in (-L, L):
            for sz in (-L, L):
                ext.append((_cell_coord(sx, v), _cell_coord(sy, v), _z_of_cell(sz)))
    rng = np.random.default_rng(17)
    base = _points(rng.uniform(-100, 100, 5000), rng.uniform(-100, 100, 5000), rng.uniform(-600, 600, 5000),
                   rng.integers(0, 1 << 24, 5000))
    edge = _points(*zip(*ext), rng.integers(0, 1 << 24, len(ext)))
    pts = np.concatenate([base, edge, edge[:3]])
    exp = rm.accumulate_downsample(pts, v, 1)
    p = abi.make_params(voxel_size=v, min_points_per_voxel=1, merge_mode=abi.MERGE_ACCUMULATE, **SMALL)
    with Pose(p) as P:
        P.trackCloudChanges(True)
        P.appendPoints(pts[:3000])
        P.appendPoints(pts[3000:])
        got = P.downsamplePtCloud().copy()
        rec, keys, counts = P.cloudChanges()
        _eq(got, exp[0])
        _eq(rec.copy(), exp[0])
        assert np.array_equal(keys, exp[1]) and np.array_equal(counts, exp[2])
        for sh in (0, 21, 42):
            f = (keys >> np.uint64(sh)) & np.uint64((1 << 21) - 1)
            assert f.min() == 1 and f.max() == (1 << 21) - 1
        bad = [(_cell_coord(L + 1, v), 0.5, 0.5), (_cell_coord(-L - 1, v), 0.5, 0.5), (0.5, _cell_coord(L + 1, v), 0.5),
               (0.5, _cell_coord(-L - 1, v), 0.5), (0.5, 0.5, _z_of_cell(L + 1)), (0.5, 0.5, _z_of_cell(-L - 1)),
               (np.nan, 0.5, 0.5), (0.5, np.nan, 0.5), (0.5, 0.5, np.nan), (np.inf, 0.5, 0.5), (0.5, -np.inf, 0.5),
               (0.5, 0.5, np.inf)]
        for q in bad:
            with pytest.raises(lib.O3RError) as e:
                P.appendPoints(np.concatenate([base[:100], _points([q[0]], [q[1]], [q[2]], [7])]))
            assert e.value.code == abi.O3R_ERR_INVALID, q
        _eq(P.downsamplePtCloud().copy(), exp[0])


# ------------------------------------------------------------------------------------ 2^30 points (RETAIN)
BIG_CHUNK = 1 << 28
BIG_TAIL = 1 << 26
BIG_N = 4 * BIG_CHUNK + BIG_TAIL
BIG_BYTES_NEEDED = 80 << 30   # cloud (grown by 1.5x), result buffer ckey, sort buffer, status words: from the buffer sizes


def _dyadic_rgb(c):
    c = np.asarray(c, np.uint32)
    return ((c % 256) << 16) | ((2 * c % 256) << 8) | (3 * c % 256)


def _big_chunk(n, seed):
    """Cell A at (0, 0, -500) fills the chunk; 300 cells x = 1..300 with dyadic coordinates, 16 points each; cell C at
    x = 301 with ~2^16 random points.  Non-A points sit at seeded positions; A's coordinates and colour are 0."""
    rng = np.random.default_rng(seed)
    pts = np.zeros(n, dtype=abi.POINT)
    pts["z"] = F32(-500.0)
    nd = 300 * 16
    nc = (1 << 16) + 123
    pos = np.unique(rng.integers(0, n, 2 * (nd + nc)))   # distinct positions, then a seeded order
    pos = rng.permutation(pos)[:nd + nc]
    dc = np.repeat(np.arange(1, 301), 16)
    d = pts[pos[:nd]]
    d["x"] = dc.astype(F32) + F32(0.5)
    d["y"] = F32(0.25)
    d["z"] = F32(-499.5)
    d["rgb"] = _dyadic_rgb(dc)
    pts[pos[:nd]] = d
    c = _points(F32(301) + rng.uniform(0.01, 0.99, nc).astype(F32), rng.uniform(0.01, 0.99, nc),
                F32(-500) + rng.uniform(0.01, 0.99, nc).astype(F32), rng.integers(0, 1 << 24, nc))
    cpos = np.sort(pos[nd:])
    pts[cpos] = c
    return pts, pts[cpos].copy()


def test_retain_2pow30_points_one_segment():
    """2^30 + 2^26 points, voxel_size 1: cell A holds more than 2^30 of them, so in both passes of the 9-bit key one
    digit's look-back prefix passes 2^30 (the 64-bit status words).  Cell A's run spans ~a million reduce tiles whose
    carries hand on serially.  Dyadic cells have closed-form records; cell C's record is the oracle's on C's points
    alone, in append order."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    free, total = torch.cuda.mem_get_info()
    name = torch.cuda.get_device_name()
    if free < BIG_BYTES_NEEDED:
        pytest.skip(f"{name}: {free / 2**30:.1f} GiB free of {total / 2**30:.1f}, the 2^30-point case needs "
                    f"{BIG_BYTES_NEEDED / 2**30:.0f} GiB")
    chunk, c_chunk = _big_chunk(BIG_CHUNK, 18)
    tail, c_tail = _big_chunk(BIG_TAIL, 19)
    p = abi.make_params(voxel_size=1.0, min_points_per_voxel=1, merge_mode=abi.MERGE_RETAIN, **SMALL)
    with Pose(p) as P:
        for _ in range(4):
            P.appendPoints(chunk)
        P.appendPoints(tail)
        assert P.cloudSize() == BIG_N
        t0 = time.perf_counter()
        got = P.downsamplePtCloud().copy()
        dt = time.perf_counter() - t0
    print(f"\n2^30 case on {name} ({free / 2**30:.1f} GiB free): {BIG_N} points -> {len(got)} records, downsample {dt:.2f} s")
    assert len(got) == 302
    a = got[0]
    assert a["x"] == 0 and a["y"] == 0 and a["z"] == F32(-500.0) and a["rgb"] == 0
    c = np.arange(1, 301)
    exp_d = _points(c.astype(F32) + F32(0.5), np.full(300, 0.25), np.full(300, -499.5), _dyadic_rgb(c))
    _eq(got[1:301], exp_d)
    c_all = np.concatenate([c_chunk] * 4 + [c_tail])
    exp_c = ob.downsample_pt_cloud(abi.make_params(voxel_size=1.0, min_points_per_voxel=1), c_all, True)
    assert len(exp_c) == 1
    _eq(got[301:], exp_c)
