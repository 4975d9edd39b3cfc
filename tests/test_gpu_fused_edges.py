"""O3R_MERGE_ACCUMULATE_FUSED's tile engine (csrc/tile.cuh) and bucket engine (csrc/bucket.cuh) at the limits they are built
around: the window radius R, the tile and halo edges, the three phase-C paths, the record-list rerun, u8 disparities whose
|q14 d + q15| is not monotone, the +-2^20 combined-cell keys both engines pack themselves, and batches of 32768 frames and
more in one chunk.

Every case compares with the oracle three ways: the per-frame VoxelGrid centroids bit for bit (as a multiset, through the
keep-frame-voxels probe) and the per-frame counts exactly; the resident combined grid (exportCells) against the exact
per-cell sums of the oracle's cloud_big (tests/reduce_model.cell_sums: keys, counts and colour sums exact, coordinate sums
within 1e-5 of the sum of their magnitudes); and the engine that served the batch.  The cases about R, a rerun flag or a
phase-C path run in a subprocess with O3R_TRACE=1 (tests/fused_edges_worker.py) and check the trace too.
"""
import ctypes as C
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle_binding as ob
import reduce_model as rm
from online_3d_reconstruction_b200 import abi, synth
from online_3d_reconstruction_b200.lib import O3RError
from online_3d_reconstruction_b200.pose import Pose

pytestmark = pytest.mark.gpu

FUSED = abi.MERGE_ACCUMULATE_FUSED
SORT, BUCKET, TILE = 0, 1, 2
FLAG_RANGE, FLAG_SPACE, FLAG_PASS = 1, 2, 4
TILE_W, TILE_H = 64, 32
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fused_edges_worker.py")
LIM = (1 << 20) - 1


# ------------------------------------------------------------------------------------------------------------ helpers
def _multiset(a):
    v = np.ascontiguousarray(a).view(np.uint32).reshape(-1, 4)
    return v[np.lexsort((v[:, 3], v[:, 2], v[:, 1], v[:, 0]))]


def _cells_match(got, ref):
    """exportCells() records against reduce_model.cell_sums of the oracle's cloud_big."""
    assert len(got) == len(ref), (len(got), len(ref))
    assert np.array_equal(got["key"], ref["key"])
    assert np.array_equal(got["n"], ref["n"])
    for f in ("sr", "sg", "sb"):
        assert np.array_equal(got[f].astype(np.uint64), ref[f]), f
    for f, a in (("sx", "ax"), ("sy", "ay"), ("sz", "az")):
        err = np.abs(got[f].astype(np.float64) - ref[f])
        lim = 1e-5 * np.maximum(ref[a], 1e-3)
        assert np.all(err <= lim), f"{f}: worst {np.max(err / lim):.3g} x the tolerance"


def _check(p, cycles, disp_type=abi.DISP_U8, engines=None, device_pointers=False, prefetch=False, host_cycles=None):
    """Oracle and GPU over the same cycles; every comparison of the module header.  -> (engines, exportCells()).
    With device pointers the oracle reads `host_cycles`, the same frames in host memory."""
    cloud, n, got_engines = None, 0, []
    with Pose(p) as P:
        P.setKeepFrameVoxels(True)
        for ci, frames in enumerate(cycles):
            at = n
            cloud, n, counts = ob.run_cycle(p, (host_cycles or cycles)[ci], disp_type, 16, cloud, n)
            if prefetch:
                got = P.createCycleClouds(P.prefetchCycle(frames, disp_type), disp_type)
            else:
                got = P.createCycleClouds(frames, disp_type, device_pointers=device_pointers)
            got_engines.append(P.lastCycleEngine())
            bad = np.nonzero(got != counts)[0]
            assert len(bad) == 0, f"{len(bad)} frame counts differ, first frame {bad[0]}: {got[bad[0]]} vs {counts[bad[0]]}"
            assert np.array_equal(_multiset(P.lastCyclePoints()), _multiset(cloud[at:n])), "per-frame voxels differ"
        cells = P.exportCells()
    _cells_match(cells, rm.cell_sums(cloud[:n], p.voxel_size))
    if engines is not None:
        assert got_engines == list(engines), (got_engines, engines)
    return got_engines, cells


def _traced(case, *args):
    """Runs a case in the worker with O3R_TRACE=1 -> one dict per fused batch: engine it started with, starting R, whether
    the bucket engine was already off, the (flags, R) of every rejected tile attempt and the (histogram / scan flags,
    reduce flags) of a rejected bucket attempt."""
    env = dict(os.environ, O3R_TRACE="1")
    r = subprocess.run([sys.executable, WORKER, case, *map(str, args)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "CASE OK" in r.stdout, (r.stdout[-3000:], r.stderr[-6000:])
    batches = []
    for line in r.stderr.splitlines():
        m = re.search(r"fused: engine (\w+) .* R (-?\d+)\)", line)
        if m:
            batches.append({"engine": m.group(1), "R": int(m.group(2)), "flags": [], "bk_flags": [],
                            "bucket_off": int(re.search(r"bucket_off (\d)", line).group(1))})
            continue
        m = re.search(r"bucket engine overflow flags (\d+) (\d+)", line)
        if m:
            batches[-1]["bk_flags"].append((int(m.group(1)), int(m.group(2))))
            continue
        m = re.search(r"tile engine flags (\d+) \(R (\d+)\)", line)
        if m:
            batches[-1]["flags"].append((int(m.group(1)), int(m.group(2))))
    assert batches, r.stderr[-3000:]
    return batches


def _final_r(b):
    """R of the tile engine's accepted attempt of a traced batch."""
    if not b["flags"]:
        return b["R"]
    fl, r = b["flags"][-1]
    return r + 1 if fl & FLAG_RANGE and not fl & FLAG_PASS else r


def _tv_radius(p, Ts):
    """Host mirror of tv_plan / tv_begin (csrc/host_tile.cuh): the window radius a context starts with."""
    Q = list(p.Q)
    ny, nx = abi.scan_dims(p)
    x0, bb, md = p.cols_start_aft_cutout, p.bounding_box, p.min_disparity
    tx = max(abs(Q[0] * x0 + Q[3]), abs(Q[0] * (x0 + nx - 1) + Q[3])) / abs(Q[11])
    ty = max(abs(Q[5] * bb + Q[7]), abs(Q[5] * (bb + ny - 1) + Q[7])) / abs(Q[11])
    rng = abs(Q[11] / (Q[14] * md + Q[15])) * math.sqrt(1 + tx * tx + ty * ty)
    T = [np.asarray(t, np.float32).reshape(4, 4).astype(np.float64) for t in Ts]
    tmax = max(float(np.abs(t[:3, 3]).max()) for t in T)
    edge = float(np.float32(p.voxel_size / 5)) * 1.001 + 16 * float(np.finfo(np.float32).eps) * (tmax + rng)
    L = 0.0
    for t in T:
        s = np.abs(np.linalg.inv(t[:3, :3])).sum(1)
        L = max(L, max((s[0] + tx * s[2]) / abs(Q[0]), (s[1] + ty * s[2]) / abs(Q[5])) * edge)
    need = abs(Q[14] * 2 * md + Q[15])
    return next((r for r in range(1, 5) if (r + 1) / L >= need), 4)


def _eye(tx=0.0, ty=0.0, tz=0.0):
    T = np.eye(4, dtype=np.float32)
    T[:3, 3] = (tx, ty, tz)
    return T


def _bgr(rng, rows, cols):
    return rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)


def _synth_cycle(seed, n, rows, cols, keep, traj_start=0):
    return [abi.make_frame(d, img, T, keep=keep) for d, img, T in synth.sequence(seed, n, rows, cols, traj_start=traj_start)]


def _pixel_cells(p, disp, T):
    """float64 reprojection of every valid pixel of a u8 frame -> (row, col, combined-grid i, j) (a stand-in for the
    leaf centroids' cells: good to a cell, which is all the phase-C path proofs below need)."""
    Q = list(p.Q)
    ys, xs = np.nonzero(disp > p.min_disparity)
    w = Q[14] * disp[ys, xs] + Q[15]
    X, Y = (Q[0] * xs + Q[3]) / w, (Q[5] * ys + Q[7]) / w
    M = np.asarray(T, np.float64).reshape(4, 4)
    wx = M[0, 0] * X + M[0, 1] * Y + M[0, 2] * Q[11] / w + M[0, 3]
    wy = M[1, 0] * X + M[1, 1] * Y + M[1, 2] * Q[11] / w + M[1, 3]
    return ys, xs, np.floor(wx / p.voxel_size).astype(np.int64), np.floor(wy / p.voxel_size).astype(np.int64)


def _tile_cell_stats(p, disp, T):
    """Per 64 x 32 tile of the scan: (cells its combined-grid box spans, occupied cells)."""
    ys, xs, ci, cj = _pixel_cells(p, disp, T)
    tile = ((ys - p.bounding_box) // TILE_H) * 1000 + (xs - p.cols_start_aft_cutout) // TILE_W
    out = []
    for t in np.unique(tile):
        s = tile == t
        i, j = ci[s], cj[s]
        out.append(((i.max() - i.min() + 1) * (j.max() - j.min() + 1), len(np.unique(i * (1 << 32) + j))))
    return np.array(out)


# ------------------------------------------------------------------------------------------------------------ tile engine
# voxel sizes at which the SMALL4 sequence starts with each window radius (_tv_radius; SMALL4's disparities stay below
# 2 min_disparity, so the first R is also the final one)
R_VOXEL = {1: 0.025, 2: 0.045, 3: 0.065, 4: 0.085}


def case_radius(R):
    R = int(R)
    keep = []
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=R_VOXEL[R], merge_mode=FUSED)
    cycles = [_synth_cycle(300 + R, 3, 128, 256, keep), _synth_cycle(310 + R, 3, 128, 256, keep, traj_start=3)]
    assert _tv_radius(p, [f.T for c in cycles for f in c]) == R
    _check(p, cycles, engines=[TILE, TILE])


@pytest.mark.parametrize("R", [1, 2, 3, 4])
def test_tile_engine_window_radius(R):
    """Each radius 1..4 is the one the batches run with (R = 4 is the 64-bit mask instantiation), with no rerun."""
    batches = _traced("case_radius", R)
    assert [b["engine"] for b in batches] == ["tile", "tile"]
    assert [_final_r(b) for b in batches] == [R, R] and not any(b["flags"] for b in batches), batches


def case_radius_rerun():
    keep = []
    rows, cols = 128, 256
    p = abi.make_params(rows=rows, cols=cols, jump_pixels=1, voxel_size=R_VOXEL[2], merge_mode=FUSED)
    seq = synth.sequence(320, 3, rows, cols)
    near = seq[1][0].copy()
    near[30:70, 60:200] = 195      # |w| = 329: beyond the 2-pixel window's reach (~280), inside the 3-pixel one's (~375)
    near[40:50, 90:110] = 196
    frames = [abi.make_frame(seq[0][0], seq[0][1], seq[0][2], keep=keep), abi.make_frame(near, seq[1][1], seq[1][2], keep=keep),
              abi.make_frame(seq[2][0], seq[2][1], seq[2][2], keep=keep)]
    _check(p, [frames[:1], frames[1:]], engines=[TILE, TILE])


def test_tile_engine_widens_r_by_one_inside_a_batch():
    """R = 2 serves the first batch; a patch at disparity 195 in the second raises TV_FLAG_RANGE once and the batch is
    rerun, and accepted, with R = 3."""
    b = _traced("case_radius_rerun")
    assert [x["engine"] for x in b] == ["tile", "tile"]
    assert b[0]["R"] == 2 and not b[0]["flags"]
    assert b[1]["R"] == 2 and b[1]["flags"] == [(FLAG_RANGE, 2)] and _final_r(b[1]) == 3, b


def _wall_frames(p, offsets, disps, keep, seed):
    """One flat fronto-parallel wall per (column offset, row offset): constant disparity, identity rotation, and a
    translation that puts a leaf boundary exactly `offset` pixels past a tile's column / row edge (half a pixel before the
    pixel, so that float rounding cannot move it)."""
    rows, cols, x0, bb = p.rows, p.cols, p.cols_start_aft_cutout, p.bounding_box
    ny, nx = abi.scan_dims(p)
    Q = list(p.Q)
    leaf = float(np.float32(p.voxel_size / 5))
    rng = np.random.default_rng(seed)
    frames = []
    for q, ((oc, orow), d) in enumerate(zip(offsets, disps)):
        w = Q[14] * d + Q[15]
        xb = x0 + (TILE_W if nx > TILE_W + oc else 0) + oc
        yb = bb + (TILE_H if ny > TILE_H + orow else 0) + orow
        tx = 1000 * leaf - (Q[0] * (xb - 0.5) + Q[3]) / w
        ty = 1000 * leaf - (Q[5] * (yb - 0.5) + Q[7]) / w
        disp = np.zeros((rows, cols), np.uint8)
        disp[bb:bb + ny, x0:x0 + nx] = d
        frames.append(abi.make_frame(disp, _bgr(rng, rows, cols), _eye(tx, ty, 3.0 + 0.01 * q), keep=keep))
    return frames


WALL_ROI = [(4, 1), (64, 32), (68, 33), (204, 33), (204, 1), (64, 33)]


@pytest.mark.parametrize("nx,ny", WALL_ROI)
def test_tile_engine_leaf_boundaries_at_tile_and_halo_edges(nx, ny):
    """Leaf boundaries 0, 1, R and 63 pixels past a tile's column edge and 0, 1 and 31 past its row edge, on ROIs 4 / 64 /
    68 / 204 pixels wide and 1 / 32 / 33 high: a leaf's first point and its mates sit in different tiles' cores, and the
    halo must show the owner every mate.  Leaves of 3-4 pixels (voxel 0.085 at disparities 115-127)."""
    keep = []
    bb, x0 = 4, 4
    p = abi.make_params(rows=ny + 2 * bb, cols=x0 + nx + bb, jump_pixels=1, voxel_size=0.085, merge_mode=FUSED, bounding_box=bb,
                        cutout_ratio=(x0 + nx + bb) // x0)
    assert p.cols_start_aft_cutout == x0 and abi.scan_dims(p) == (ny, nx)
    R = _tv_radius(p, [_eye()])
    offs = [(oc, orow) for oc in (0, 1, R, 63) for orow in (0, 1, 31)]
    frames = _wall_frames(p, offs, [115 + (q % 13) for q in range(len(offs))], keep, seed=nx * 100 + ny)
    # one batch: on the narrowest ROIs a frame holds a leaf or two, too few to reduce, and the context would leave the engine
    _check(p, [frames], engines=[TILE])


def _two_wall_frame(p, keep, seed, d_even, d_odd):
    rows, cols, x0, bb = p.rows, p.cols, p.cols_start_aft_cutout, p.bounding_box
    disp = np.zeros((rows, cols), np.uint8)
    disp[:, :] = d_even
    disp[:, 1::2] = d_odd
    disp[:bb], disp[rows - bb:], disp[:, :x0] = 0, 0, 0
    return disp, abi.make_frame(disp, _bgr(np.random.default_rng(seed), rows, cols), _eye(0.2, -0.1, 1.0), keep=keep)


def test_tile_engine_sparse_hash_cells_are_exact_and_reproducible():
    """Columns alternate between disparities 66 and 126 (depths 38 m and 20 m) inside every tile: a tile's combined-grid
    box spans far more cells than the 512-cell dense table, while fewer than 512 are occupied — phase C numbers the cells
    through the open-addressing hash, whose numbering depends on an atomic race.  Exact against the oracle, and two
    contexts give bit-identical exportCells()."""
    keep = []
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED)
    disp, fr = _two_wall_frame(p, keep, 1, 66, 126)
    st = _tile_cell_stats(p, disp, fr.T)
    assert st[:, 0].min() > 1024 and st[:, 1].max() < 256, st
    _, a = _check(p, [[fr]], engines=[TILE])
    _, b = _check(p, [[fr]], engines=[TILE])
    assert a.tobytes() == b.tobytes()


def test_tile_engine_loose_path_when_a_tile_occupies_more_than_512_cells():
    """voxel 0.005 against a pixel footprint of 9 mm (disparity 66): every centroid of a tile is alone in its combined cell,
    more than 512 per tile — phase C's single-point records."""
    keep = []
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=0.005, merge_mode=FUSED)
    disp, fr = _two_wall_frame(p, keep, 2, 66, 66)
    st = _tile_cell_stats(p, disp, fr.T)
    assert st[:, 1].max() > 1024, st
    _check(p, [[fr]], engines=[TILE])


def case_record_growth():
    keep = []
    rows, cols = 128, 256
    p = abi.make_params(rows=rows, cols=cols, jump_pixels=1, voxel_size=0.013, merge_mode=FUSED)
    rng = np.random.default_rng(5)
    small = np.zeros((rows, cols), np.uint8)
    small[40:50, 100:110] = 100
    wall = np.zeros((rows, cols), np.uint8)
    wall[p.bounding_box:rows - p.bounding_box, p.cols_start_aft_cutout:cols - p.bounding_box] = 100
    first = [abi.make_frame(small, _bgr(rng, rows, cols), _eye(0.0, 0.0, 1.0), keep=keep)]
    dense = [abi.make_frame(wall, _bgr(rng, rows, cols), _eye(0.003 * q, 0.002 * q, 1.0), keep=keep) for q in range(2)]
    st = _tile_cell_stats(p, wall, dense[0].T)
    assert st[:, 1].sum() > 256 * len(st) and (88 * 204) / st[:, 1].sum() > 4, st   # > 256 records a tile, a 4x reduction
    more = [abi.make_frame(wall, _bgr(rng, rows, cols), _eye(0.001, 0.004, 1.0), keep=keep)]
    _check(p, [first, dense, more], engines=[TILE, TILE, TILE])


def test_tile_engine_grows_its_record_lists_and_reruns():
    """A first batch sizes the record lists for 256 records a tile; a later batch of dense walls needs ~350 a tile (and still
    reduces 5x): TV_FLAG_SPACE, the lists grow to what the device reported, the batch is rerun exactly, and the engine stays."""
    b = _traced("case_record_growth")
    assert [x["engine"] for x in b] == ["tile"] * 3
    # (the first batch may rerun once on PCL's pass-through guess: its leaf is small against the nominal frustum)
    assert not any(f & FLAG_SPACE for f, _ in b[0]["flags"]), b
    assert b[1]["flags"] and all(f & FLAG_SPACE for f, _ in b[1]["flags"]), b
    assert not b[2]["flags"], b


def _lut_frames(p, keep, lo, hi, disp_type):
    """Smooth disparity fields covering [lo, hi] (never 200.5, where w = 0), each frame also as f32."""
    rows, cols = p.rows, p.cols
    rng = np.random.default_rng(lo * 1000 + hi)
    yy, xx = np.mgrid[0:rows, 0:cols]
    out = []
    for q, (_, img, T) in enumerate(synth.sequence(330 + lo, 3, rows, cols)):
        f = lo + (hi - lo) * (0.5 + 0.5 * np.sin(xx / (9.0 + 3 * q) + yy / 23.0 + q))
        d = np.clip(np.rint(f + rng.normal(0, 0.7, f.shape)), lo, hi).astype(np.uint8)
        d[:, : cols // 8] = 0
        out.append(abi.make_frame(d.astype(abi.DISP_NP[disp_type]), img, T, keep=keep))
    return out


@pytest.mark.parametrize("lo,hi", [(65, 150), (65, 255)])
@pytest.mark.parametrize("disp_type", [abi.DISP_U8, abi.DISP_F32])
def test_nonmonotone_w_u8_lut_and_f32(lo, hi, disp_type):
    """Q[15] = -200.5 Q[14]: w = q14 (d - 200.5) has the same sign at min_disparity and at twice it, so the tile engine
    accepts the Q, but |w| FALLS from 228 at d = 65 to 0 at 200.5 and rises again.  The u8 path checks the window through
    the largest passing disparity instead of |w| per pixel; low disparities, whose |w| is above the bound, must still raise
    the range flag.  The same frames as f32 take the per-pixel check.  Whichever engine serves them, exact."""
    keep = []
    q = list(abi.Q_CAM13)
    q[15] = -200.5 * q[14]
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, Q=tuple(q))
    _check(p, [_lut_frames(p, keep, lo, hi, disp_type)], disp_type=disp_type)


# ------------------------------------------------------------------------------------------------------------ +-2^20 cells
def _limit_frame(p, keep, tx, ty, d):
    rows, cols = p.rows, p.cols
    disp = np.zeros((rows, cols), np.uint8)
    disp[40:48, 60:72] = d
    disp[44, 64:68] = d + 1
    return abi.make_frame(disp, _bgr(np.random.default_rng(d), rows, cols), _eye(tx, ty, 2.0), keep=keep)


def _place(p, keep, d, axis, edge_cell):
    """A patch frame whose combined cells reach exactly `edge_cell` on `axis` (0 = x, 1 = y: the largest cell when it is
    positive, the smallest when negative), found from the oracle's voxel centroids."""
    v = p.voxel_size
    t = [0.0, 0.0]
    for _ in range(8):
        fr = _limit_frame(p, keep, t[0], t[1], d)
        cloud, n, _ = ob.run_cycle(p, [fr], abi.DISP_U8, 1)
        c = rm.cells(cloud[:n], v)[axis]
        edge = c.max() if edge_cell > 0 else c.min()
        if edge == edge_cell:
            return fr
        t[axis] += (edge_cell - edge) * v
    raise AssertionError(f"no translation puts the patch on cell {edge_cell} (reached {edge})")


@pytest.mark.parametrize("engine", [TILE, BUCKET])
def test_combined_cell_limit_through_the_frames_path(engine):
    """Frames whose points sit on combined cell +-(2^20 - 1) of x / y are accepted and exact; at +-2^20, where the 21-bit
    key field wraps, the batch is refused with O3R_ERR_INVALID and the resident map is bitwise unchanged — the engines pack 21-bit key fields before the
    host checks the range, so a wrapped key must never reach the map.  Disparity 6 over min_disparity 4: far enough that
    the tile engine's window holds the float rounding of 52 km coordinates.  (The z axis is not covered: its cells are
    1000 high, and z = +-2^20 cells lies beyond what either fused engine accepts.)"""
    keep = []
    geom = dict(rows=128, cols=256) if engine == TILE else dict(rows=120, cols=200)
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, min_disparity=4.0, **geom)
    ok, over = [], []
    for axis in (0, 1):
        for sign in (1, -1):
            ok.append(_place(p, keep, 6, axis, sign * LIM))
            over.append(_place(p, keep, 6, axis, sign * (LIM + 1)))
    _, cells = _check(p, [ok], engines=[engine])
    keys = cells["key"].astype(np.uint64)
    ci = (keys & np.uint64((1 << 21) - 1)).astype(np.int64) - (1 << 20)
    cj = ((keys >> np.uint64(21)) & np.uint64((1 << 21) - 1)).astype(np.int64) - (1 << 20)
    assert ci.max() == LIM and ci.min() == -LIM and cj.max() == LIM and cj.min() == -LIM
    with Pose(p) as P:
        P.createCycleClouds(ok)
        before = P.exportCells()
        assert P.lastCycleEngine() == engine
        for fr in over:
            with pytest.raises(O3RError) as e:
                P.createCycleClouds([fr])
            assert "2^20" in str(e.value)
            assert P.exportCells().tobytes() == before.tobytes()


# ------------------------------------------------------------------------------------------------------------ bucket engine
# cutout_ratio 8: ROI 31 x 16 from column 5, rows not 4-aligned -> bucket engine; cutout_ratio 10: ROI 32 x 16 from column 4
# -> tile engine
TINY = dict(rows=24, cols=40, bounding_box=4, min_disparity=110.0)
N_IMG = 16


def _tiny_images(p, seed):
    """N_IMG tiny frames: a patch of a few hundred pixels at disparities 118-126 (leaves of 2-4 points)."""
    rng = np.random.default_rng(seed)
    d = np.zeros((N_IMG, p.rows, p.cols), np.uint8)
    for q in range(N_IMG):
        h, w = 8 + q % 5, 18 + q % 9
        d[q, 6:6 + h, 10:10 + w] = rng.integers(118, 127, (h, w), dtype=np.uint8)
    return d, rng.integers(0, 256, (N_IMG, p.rows, p.cols, 3), dtype=np.uint8)


def _tiny_T(i):
    return _eye(0.37 * (i % 97) + 0.011 * (i // 97), -0.23 * (i % 89), 1.0 + 0.001 * (i % 7))


def _many_frames(p, n, dev, keep, seed):
    import torch
    d, img = _tiny_images(p, seed)
    if dev:
        dd, di = torch.from_numpy(d).cuda(), torch.from_numpy(img).cuda()
        keep.extend([dd, di])
    host, frames = [], []
    for i in range(n):
        q = i % N_IMG
        host.append(abi.make_frame(d[q], img[q], _tiny_T(i), keep=keep))
        fr = abi.make_frame(d[q], img[q], _tiny_T(i), keep=keep)
        if dev:
            fr.disp, fr.bgr = dd[q].data_ptr(), di[q].data_ptr()
        frames.append(fr)
    return frames, host


@pytest.mark.parametrize("n,how,engine", [(32769, "device", BUCKET), (65535, "device", BUCKET), (32769, "prefetch", BUCKET),
                                          (32769, "device", TILE)])
def test_bucket_engine_batches_of_32768_frames_and_more(n, how, engine):
    """Device-pointer and prefetched batches run as ONE chunk, so the bucket engine's chunk-local frame index reaches 65534:
    frames 32768 and up must keep their own per-frame counts and voxels (not be mistaken for PCL pass-through frames of
    frame f - 32768).  The tile engine at the same size is the control."""
    pytest.importorskip("torch")
    keep = []
    geom = dict(TINY, cutout_ratio=8 if engine == BUCKET else 10)
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, max_batch_frames=65535, **geom)
    frames, host = _many_frames(p, n, how == "device", keep, seed=n)
    _check(p, [frames], engines=[engine], device_pointers=how == "device", prefetch=how == "prefetch", host_cycles=[host])


# One case per limit of the bucket engine.  Each runs traced: the first batch starts on the bucket engine (unaligned rows
# keep the tile engine out), and the trace shows the device's flags — histogram / scan word (2 = a bucket above kBkCapSlow),
# reduce word (2 = a bucket larger than one reduce CTA holds, 4 = too many strays) — or that none was raised.
BK_BUCKET, BK_PART = 2, 4


def case_bucket_over_reduce_cta():
    keep = []
    p = abi.make_params(rows=120, cols=200, jump_pixels=1, voxel_size=0.5, merge_mode=FUSED)
    _check(p, [_synth_cycle(340, 2, 120, 200, keep), _synth_cycle(341, 2, 120, 200, keep, traj_start=2)], engines=[SORT, SORT])


def test_bucket_engine_falls_back_when_a_bucket_outgrows_the_reduce():
    """voxel 0.5: buckets of several thousand points, more than one reduce CTA holds (kRdCap): the reduce flags it, this
    batch is rerun through the sort engine and the context stays there — exact either way."""
    b = _traced("case_bucket_over_reduce_cta")
    assert [x["engine"] for x in b] == ["bucket", "sort"] and b[1]["bucket_off"] == 1, b
    (h, r), = b[0]["bk_flags"]
    assert h == 0 and r & BK_BUCKET, b


def _wall(p, d):
    disp = np.zeros((p.rows, p.cols), np.uint8)
    ny, nx = abi.scan_dims(p)
    disp[p.bounding_box:p.bounding_box + ny, p.cols_start_aft_cutout:p.cols_start_aft_cutout + nx] = d
    return disp


def case_bucket_over_capslow():
    keep = []
    p = abi.make_params(rows=240, cols=330, jump_pixels=1, voxel_size=5.0, merge_mode=FUSED, bounding_box=4)
    assert np.prod(abi.scan_dims(p)) > 65535
    # a wall at disparity 100 moved into combined cell (0, 0): every point in one 5 m bucket
    fr = abi.make_frame(_wall(p, 100), _bgr(np.random.default_rng(7), p.rows, p.cols), _eye(3.0, 3.1, 1.0), keep=keep)
    _check(p, [[fr]], engines=[SORT])


def test_bucket_engine_falls_back_when_a_bucket_passes_kbkcapslow():
    """66 120 points of one frame in one bucket (voxel 5 m), more than a bucket's 16-bit count holds: the histogram raises
    its flag, the later passes skip, and the batch is rerun through the sort engine — exact."""
    b = _traced("case_bucket_over_capslow")
    assert [x["engine"] for x in b] == ["bucket"] and b[0]["bk_flags"] == [(BK_BUCKET, 0)], b


def _side_T(p, d, z_row, row):
    """Camera looking sideways: world x = camera x, world y = depth, world z = -camera y.  A fronto-parallel wall at
    disparity d then stands at one world y, and a bucket (5 x 5 leaf columns in x, y) holds a vertical stripe of it, all rows.
    The translation puts pixel row `row` at world z = z_row and the wall at world y = 0.025 (mid-leaf)."""
    Q = list(p.Q)
    w = Q[14] * d + Q[15]
    T = np.array([[1, 0, 0, 0.2], [0, 0, 1, 0], [0, -1, 0, 0], [0, 0, 0, 1]], dtype=np.float64)
    T[1, 3] = 0.025 - Q[11] / w
    T[2, 3] = z_row + (Q[5] * row + Q[7]) / w
    return T.astype(np.float32)


def case_bucket_strays_in_one_bucket():
    keep = []
    p = abi.make_params(rows=120, cols=200, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED)
    # the combined grid's z boundary (z + 500 = 1000) halfway down the wall: in every bucket the leaves above it land in
    # another combined cell than the bucket's nominal one — some 20 strays per bucket
    fr = abi.make_frame(_wall(p, 100), _bgr(np.random.default_rng(8), p.rows, p.cols), _side_T(p, 100, 500.003, 60), keep=keep)
    cloud, n, counts = ob.run_cycle(p, [fr], abi.DISP_U8, 1)
    assert counts[0] < 8192   # fewer centroids than the chunk's stray cap: only the per-bucket limit can fire
    _check(p, [[fr]], engines=[SORT])


def test_bucket_engine_falls_back_on_more_than_krdstray_strays_in_a_bucket():
    b = _traced("case_bucket_strays_in_one_bucket")
    assert [x["engine"] for x in b] == ["bucket"] and b[0]["bk_flags"] == [(0, BK_PART)], b


def _stray_frames(p, n, keep):
    """Walls of pixel columns 10 apart (at most two in a bucket) whose top row alone lies above the z boundary: one stray
    per column, ~90 per frame."""
    disp = np.zeros((p.rows, p.cols), np.uint8)
    ny, nx = abi.scan_dims(p)
    x0, bb = p.cols_start_aft_cutout, p.bounding_box
    disp[bb:bb + ny, x0:x0 + nx:10] = 100
    rng = np.random.default_rng(9)
    return [abi.make_frame(disp, _bgr(rng, p.rows, p.cols), _side_T(p, 100, 500.003 + 0.0001 * (i % 3), bb), keep=keep)
            for i in range(n)]


def case_bucket_chunk_stray_cap(how):
    import torch
    keep = []
    p = abi.make_params(rows=24, cols=1032, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, bounding_box=4, max_batch_frames=120)
    host = _stray_frames(p, 120, keep)
    if how == "host":   # chunks of 10 frames: ~900 strays a chunk
        _check(p, [host], engines=[BUCKET])
        return
    frames = []
    for fr in host:   # one chunk of 120 frames: ~10 800 strays, past the 8192 a chunk keeps
        d = torch.from_numpy(np.ctypeslib.as_array((C.c_uint8 * (p.rows * fr.disp_step)).from_address(fr.disp)).copy()).cuda()
        c = torch.from_numpy(np.ctypeslib.as_array((C.c_uint8 * (p.rows * fr.bgr_step)).from_address(fr.bgr)).copy()).cuda()
        keep.extend([d, c])
        g = abi.Frame.from_buffer_copy(fr)
        g.disp, g.bgr = d.data_ptr(), c.data_ptr()
        frames.append(g)
    _check(p, [frames], engines=[SORT], device_pointers=True, host_cycles=[host])


@pytest.mark.parametrize("how", ["host", "device"])
def test_bucket_engine_chunk_stray_cap(how):
    """At most 8192 stray records a chunk (kBkStrayCap).  120 frames of ~90 strays each, never more than two in a bucket: in
    host chunks of 10 frames the bucket engine serves them; as one device-pointer chunk the reduce raises its stray flag
    and the batch is rerun through the sort engine.  Exact both ways."""
    pytest.importorskip("torch")
    b = _traced("case_bucket_chunk_stray_cap", how)
    assert [x["engine"] for x in b] == ["bucket"], b
    assert b[0]["bk_flags"] == ([] if how == "host" else [(0, BK_PART)]), b


def case_bucket_grid_unbounded():
    keep = []
    p = abi.make_params(rows=120, cols=200, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED)
    cycles = [[abi.make_frame(d, img, _eye(0.0, 0.0, 1.0e5), keep=keep) for d, img, _ in synth.sequence(343, 2, 120, 200)]]
    _check(p, cycles, engines=[SORT])


def test_bucket_engine_refuses_a_frame_grid_it_cannot_bound():
    """z = 100 km over 1 cm leaves: the frame's leaf cells pass the 8e6 the bucket grid keeps float cell arithmetic exact
    for (and with it any z range near 2^26 leaf cells, kBkKBits), so the host never starts the bucket engine: the batch runs
    the sort engine from the start, no overflow flag, exact."""
    b = _traced("case_bucket_grid_unbounded")
    assert [(x["engine"], x["bucket_off"], x["bk_flags"]) for x in b] == [("sort", 0, [])], b


def test_bucket_engine_big_buckets_are_served():
    """voxel 0.12 on unaligned rows: several hundred points in one 5 x 5-leaf bucket, ranked inside their (bucket, leaf
    column) bins — served by the bucket engine, exact."""
    keep = []
    p = abi.make_params(rows=120, cols=200, jump_pixels=1, voxel_size=0.12, merge_mode=FUSED)
    _check(p, [_synth_cycle(342, 3, 120, 200, keep)], engines=[BUCKET])
