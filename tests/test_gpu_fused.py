"""GPU parity of O3R_MERGE_ACCUMULATE_FUSED (the mode bench.py times) against the CPU oracle, through the C-ABI, from small
ragged cases up to BASELINE.json's configs at full size.  Three engines serve the mode (o3r_last_batch_engine): the tile
engine (csrc/tile.cuh: dense scans of a rectified-stereo Q), the bucket engine (csrc/bucket.cuh: strided scans, keypoints,
geometries without aligned rows, leaves wider than the tile engine's pixel window) and the sort engine (everything else).

Contract (include/o3r.h): per-frame VoxelGrid centroids bit-identical to the oracle's (checked as a multiset through the
keep-frame-voxels probe, because the fused engine never materialises the per-frame clouds in order), per-frame voxel
counts exact, combined-grid cells / order / counts / colours exact, combined centroids within 1e-5 relative (float
reassociation of the per-cell partial sums), results reproducible bit for bit.
"""
import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi, synth
from online_3d_reconstruction_b200.pose import Pose
from test_gpu_parity import SMALL, SMALL4, _close, _eq, _frames

pytestmark = pytest.mark.gpu

FUSED = abi.MERGE_ACCUMULATE_FUSED
SORT, BUCKET, TILE = 0, 1, 2


def _multiset(a):
    """Records as sorted raw 128-bit values: order-free bitwise comparison."""
    v = np.ascontiguousarray(a).view(np.uint32).reshape(-1, 4)
    return v[np.lexsort((v[:, 3], v[:, 2], v[:, 1], v[:, 0]))]


def _run_cycles(p, cycles, disp_type=abi.DISP_U8, expect_engine=TILE, probe=True, threads=4):
    """Oracle and GPU over the same cycles -> (got combined cloud, expected combined cloud)."""
    cloud, n = None, 0
    with Pose(p) as P:
        if probe:
            P.setKeepFrameVoxels(True)
        for ci, frames in enumerate(cycles):
            at = n
            cloud, n, counts = ob.run_cycle(p, frames, disp_type, threads, cloud, n)
            got_counts = P.createCycleClouds(frames, disp_type)
            want = expect_engine[ci] if isinstance(expect_engine, (list, tuple)) else expect_engine
            assert P.lastCycleEngine() == want, (ci, P.lastCycleEngine(), want)
            assert np.array_equal(got_counts, counts), (got_counts, counts)
            if probe:   # every per-frame voxel centroid of the cycle, bit for bit (order is not defined in this mode)
                assert np.array_equal(_multiset(P.lastCyclePoints()), _multiset(cloud[at:n]))
        got = P.downsamplePtCloud()
    exp = ob.downsample_pt_cloud(p, cloud[:n], True)
    return got, exp


def _same_cells(got, exp, voxel):
    inv = np.float32(1.0) / np.float32(voxel)
    for f in ("x", "y"):
        assert np.array_equal(np.floor(got[f] * inv), np.floor(exp[f] * inv))


@pytest.mark.parametrize("min_pts", [1, 2, 5])
@pytest.mark.parametrize("geom", [SMALL, SMALL4])
def test_fused_three_cycles_small(min_pts, geom):
    keep = []
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=min_pts, merge_mode=FUSED, **geom)
    cycles = [_frames(240, 4, geom["rows"], geom["cols"], keep=keep, traj_start=0),
              _frames(241, 3, geom["rows"], geom["cols"], keep=keep, traj_start=4),
              _frames(242, 4, geom["rows"], geom["cols"], keep=keep, traj_start=5)]
    got, exp = _run_cycles(p, cycles, expect_engine=TILE if geom is SMALL4 else BUCKET)   # SMALL: rows not 4-aligned
    assert len(exp) > 50
    _close(got, exp)
    _same_cells(got, exp, 0.05)


def test_fused_unsupported_last_cycle_points_without_probe():
    from online_3d_reconstruction_b200.lib import O3RError
    keep = []
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, **SMALL4)
    with Pose(p) as P:
        P.createCycleClouds(_frames(243, 2, SMALL4["rows"], SMALL4["cols"], keep=keep))
        assert P.lastCycleEngine() == TILE
        with pytest.raises(O3RError):
            P.lastCyclePoints()
        # a single-frame call always runs the sort engine and returns the ordered per-frame cloud
        fr = _frames(243, 1, SMALL4["rows"], SMALL4["cols"], keep=keep)[0]
        _eq(P.createAndTransformPtCloud(fr), ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8))


@pytest.mark.parametrize("J,n_kp", [(3, 700), (2, 0), (15, 1500), (0, 900)])
def test_fused_strided_scan_and_keypoints(J, n_kp):
    """Keypoints first (ORB order, duplicates allowed), then the strided grid: scan positions drive the fold order."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=J, voxel_size=0.05, merge_mode=FUSED, **geom)
    cycles = [_frames(250 + J, 5, geom["rows"], geom["cols"], keep=keep, n_kp=n_kp)]
    got, exp = _run_cycles(p, cycles, expect_engine=BUCKET)
    assert len(exp) > 20
    _close(got, exp)


@pytest.mark.parametrize("disp_type", [abi.DISP_U16, abi.DISP_F32, abi.DISP_F64])
def test_fused_other_disparity_types(disp_type):
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, disp_divisor=200.0, **geom)
    cycles = [_frames(260, 3, geom["rows"], geom["cols"], disp_type=disp_type, keep=keep)]
    got, exp = _run_cycles(p, cycles, disp_type)
    assert len(exp) > 50
    _close(got, exp)


def test_fused_ragged_cycle_with_empty_and_tiny_frames():
    keep = []
    geom = SMALL4
    rows, cols = geom["rows"], geom["cols"]
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, **geom)
    frames = _frames(270, 4, rows, cols, keep=keep)
    seq = synth.sequence(270, 4, rows, cols)
    empty = abi.make_frame(np.zeros((rows, cols), np.uint8), seq[1][1], seq[1][2], keep=keep)
    tiny_d = np.zeros((rows, cols), np.uint8)
    tiny_d[40:44, 100:107] = 110
    tiny = abi.make_frame(tiny_d, seq[2][1], seq[2][2], keep=keep)
    got, exp = _run_cycles(p, [[frames[0], empty, tiny, frames[3]], [empty], [empty, tiny]])
    _close(got, exp)
    with Pose(p) as P:   # a context that never sees a valid pixel
        assert P.createCycleClouds([empty, empty]).tolist() == [0, 0]
        assert len(P.downsamplePtCloud()) == 0


def test_fused_passthrough_frames():
    """Leaf so small that PCL's int32 guard returns the per-frame cloud unchanged (what config 5 does at 4K).  At this pixel
    footprint (5.5 mm against a 2 mm combined grid) nearly every point is its own cell: the tile engine's first batch grows its
    record lists once (the device reports what it needs), reduces nothing, and the context moves on to the sort engine."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.002, merge_mode=FUSED, **geom)
    cycles = [_frames(280, 2, geom["rows"], geom["cols"], keep=keep), _frames(281, 2, geom["rows"], geom["cols"], keep=keep, traj_start=2)]
    got, exp = _run_cycles(p, cycles, expect_engine=[TILE, SORT])
    assert len(exp) > 1000
    _close(got, exp)


def test_fused_tile_engine_mixed_passthrough_and_grouped_frames():
    """One batch holds frames on both sides of PCL's int32 guard (a full frame at leaf 0.0004 trips it, a frame with a
    4 x 7 pixel patch does not): the tile kernel runs on the host's guess, the exact bboxes contradict it, and the batch is
    rerun with the guard's actual verdicts — per-frame clouds still bit-exact."""
    keep = []
    geom = SMALL4
    rows, cols = geom["rows"], geom["cols"]
    p = abi.make_params(jump_pixels=1, voxel_size=0.002, merge_mode=FUSED, **geom)
    frames = _frames(282, 3, rows, cols, keep=keep)
    seq = synth.sequence(282, 3, rows, cols)
    tiny_d = np.zeros((rows, cols), np.uint8)
    tiny_d[40:44, 100:107] = 110
    tiny_d[41, 101:104] = 111
    tiny = abi.make_frame(tiny_d, seq[1][1], seq[1][2], keep=keep)
    got, exp = _run_cycles(p, [[frames[0], tiny, frames[2]], [tiny, tiny], [frames[1]]], expect_engine=[TILE, SORT, SORT])
    _close(got, exp)


@pytest.mark.parametrize("voxel,engine", [(0.03, TILE), (0.07, TILE), (0.12, BUCKET)])
def test_fused_tile_engine_window_follows_the_leaf_size(voxel, engine):
    """The pixel window that holds a leaf's points grows with the leaf (tile.cuh): voxel_size 0.03 needs 1 pixel at these
    depths, 0.07 needs 3, at 0.12 the device reports disparities beyond even the widest window's reach (4) and the context
    moves to the bucket engine.  Same bit-exact per-frame centroids everywhere."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=voxel, merge_mode=FUSED, **geom)
    cycles = [_frames(285, 3, geom["rows"], geom["cols"], keep=keep), _frames(286, 3, geom["rows"], geom["cols"], keep=keep, traj_start=3)]
    got, exp = _run_cycles(p, cycles, expect_engine=engine)
    _close(got, exp)
    _same_cells(got, exp, voxel)


def test_fused_tile_engine_widens_its_window_when_a_disparity_is_out_of_reach():
    """voxel_size 0.05 starts with a 2-pixel window (good for disparities below ~150 in this geometry); a patch at disparity
    170 makes the device raise the range flag, the batch is rerun with 3 pixels and the context keeps that window."""
    keep = []
    geom = SMALL4
    rows, cols = geom["rows"], geom["cols"]
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, **geom)
    seq = synth.sequence(287, 4, rows, cols)
    near = seq[1][0].copy()
    near[30:60, 80:150] = 170
    near[33:40, 90:100] = 171
    cycles = [[abi.make_frame(seq[0][0], seq[0][1], seq[0][2], keep=keep)],
              [abi.make_frame(near, seq[1][1], seq[1][2], keep=keep), abi.make_frame(seq[2][0], seq[2][1], seq[2][2], keep=keep)],
              [abi.make_frame(seq[3][0], seq[3][1], seq[3][2], keep=keep)]]
    got, exp = _run_cycles(p, cycles)
    _close(got, exp)


@pytest.mark.parametrize("voxel", [0.12])
def test_fused_big_buckets_are_ranked_column_by_column(voxel):
    """voxel_size 0.12: a leaf spans more pixels than the tile engine's widest window (the device raises the range flag
    on the first batch and the context moves to the bucket engine), and several hundred points fall into one 5x5-leaf bucket:
    the reduce ranks every point inside its (bucket, leaf column) bin — PCL's order is column-major inside a bucket — same
    bit-exact per-frame centroids."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=voxel, merge_mode=FUSED, **geom)
    cycles = [_frames(290, 3, geom["rows"], geom["cols"], keep=keep), _frames(291, 3, geom["rows"], geom["cols"], keep=keep, traj_start=3)]
    got, exp = _run_cycles(p, cycles, expect_engine=BUCKET)
    _close(got, exp)
    _same_cells(got, exp, voxel)


def test_fused_falls_back_to_the_sort_engine_when_a_leaf_column_overflows():
    """voxel_size 0.5 puts ~330 points into ONE leaf column (> 128): the device raises the overflow flag, the batch is rerun
    through the sort engine (TILED contract) and the context stays there."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.5, merge_mode=FUSED, **geom)
    cycles = [_frames(292, 3, geom["rows"], geom["cols"], keep=keep), _frames(293, 3, geom["rows"], geom["cols"], keep=keep, traj_start=3)]
    got, exp = _run_cycles(p, cycles, expect_engine=SORT, probe=False)
    _close(got, exp)
    _same_cells(got, exp, 0.5)


def test_fused_generic_q_runs_the_sort_engine():
    keep = []
    geom = SMALL4
    q = list(abi.Q_CAM13)
    q[1] = 1e-3   # not the rectified-stereo sparsity: no frustum bound, the bucket engine does not apply
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, Q=tuple(q), **geom)
    got, exp = _run_cycles(p, [_frames(295, 3, geom["rows"], geom["cols"], keep=keep)], expect_engine=SORT, probe=False)
    _close(got, exp)


def test_fused_is_reproducible_and_matches_exact_mode_cells():
    keep = []
    geom = SMALL4
    frames = _frames(300, 6, geom["rows"], geom["cols"], keep=keep)
    outs = []
    for mode in (FUSED, FUSED, abi.MERGE_ACCUMULATE):
        p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=mode, **geom)
        with Pose(p) as P:
            P.createCycleClouds(frames[:3])
            P.createCycleClouds(frames[3:])
            outs.append(P.downsamplePtCloud())
    _eq(outs[0], outs[1])
    _close(outs[0], outs[2])


def test_fused_prefetch_and_chunked_host_inputs_agree_with_device_inputs():
    torch = pytest.importorskip("torch")
    keep = []
    geom = SMALL4
    rows, cols = geom["rows"], geom["cols"]
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, max_batch_frames=16, **geom)
    seq = synth.sequence(310, 14, rows, cols)
    host = [abi.make_frame(d, img, T, keep=keep) for d, img, T in seq]
    dd = [torch.from_numpy(np.ascontiguousarray(d)).cuda() for d, _, _ in seq]
    di = [torch.from_numpy(np.ascontiguousarray(img)).cuda() for _, img, _ in seq]
    dev = []
    for (d, img, T), a, b in zip(seq, dd, di):
        fr = abi.make_frame(d, img, T, keep=keep)
        fr.disp, fr.bgr = a.data_ptr(), b.data_ptr()
        dev.append(fr)
    with Pose(p) as A, Pose(p) as B, Pose(p) as Cx:
        ca = A.createCycleClouds(host)                       # chunked copies (10 + 4 frames)
        cb = B.createCycleClouds(dev, device_pointers=True)  # one launch sequence
        arr = Cx.prefetchCycle(host)
        cc = Cx.createCycleClouds(arr)                       # prefetched
        assert A.lastCycleEngine() == B.lastCycleEngine() == Cx.lastCycleEngine() == TILE
        assert np.array_equal(ca, cb) and np.array_equal(ca, cc)
        a, b, c = A.downsamplePtCloud(), B.downsamplePtCloud(), Cx.downsamplePtCloud()
    # chunking changes which frames share a launch, not any sum: partial cells are per tile and per frame
    _eq(a, b)
    _eq(a, c)


# ------------------------------------------------------------------------------ BASELINE.json configs at full size
def test_config2_full_size_50_frames_3_cycles_against_oracle():
    """BASELINE configs[1] exactly as bench.py runs it: 1280x720 u8, jump_pixels 1, voxel_size 0.05, min_points 1, 50 frames
    per cycle, three cycles, FUSED — against the oracle's run_cycle + downsamplePtCloud (pose.cpp:361-434, :527-531)."""
    keep = []
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=1, merge_mode=FUSED, max_batch_frames=50)
    seq = synth.sequence(1002, 50, 720, 1280)
    Ts = synth.trajectory(np.random.default_rng(1002 + 7919), 150)
    cycles = [[abi.make_frame(seq[i][0], seq[i][1], Ts[c * 50 + i], keep=keep) for i in range(50)] for c in range(3)]
    got, exp = _run_cycles(p, cycles, threads=16)
    assert len(exp) > 50000
    _close(got, exp)
    _same_cells(got, exp, 0.05)


def test_config4_v002_against_oracle():
    """BASELINE configs[3] geometry: voxel_size 0.02 (leaf 0.004 < pixel footprint: nearly one voxel per point, the
    per-frame int32 guard close to tripping), 12 frames per cycle, two cycles."""
    keep = []
    p = abi.make_params(jump_pixels=1, voxel_size=0.02, min_points_per_voxel=1, merge_mode=FUSED, max_batch_frames=12)
    seq = synth.sequence(1004, 12, 720, 1280)
    Ts = synth.trajectory(np.random.default_rng(1004 + 7919), 24)
    cycles = [[abi.make_frame(seq[i][0], seq[i][1], Ts[c * 12 + i], keep=keep) for i in range(12)] for c in range(2)]
    got, exp = _run_cycles(p, cycles, threads=16)
    assert len(exp) > 100000
    _close(got, exp)
    _same_cells(got, exp, 0.02)


def test_config5_4k_u16_passthrough_against_oracle():
    """BASELINE configs[4] geometry: 3840x2160 u16 disparity / 200, voxel_size 0.01: the per-frame grid overflows int32 and
    PCL passes the frame through; combined grid at 0.01.  Two frames per cycle, two cycles."""
    keep = []
    p = abi.make_params(rows=2160, cols=3840, jump_pixels=1, voxel_size=0.01, min_points_per_voxel=1, merge_mode=FUSED,
                        Q=synth.q_scaled(3.0), disp_divisor=200.0, max_batch_frames=2)
    seq = synth.sequence(1005, 2, 2160, 3840, disp_type=abi.DISP_U16)
    Ts = synth.trajectory(np.random.default_rng(1005 + 7919), 4)
    cycles = [[abi.make_frame(seq[i][0], seq[i][1], Ts[c * 2 + i], keep=keep) for i in range(2)] for c in range(2)]
    # 5.5 mm between neighbouring points, ~0.6 m of depth noise scattering them sideways, a 1 cm combined grid: a 64 x 32 tile
    # spreads its 2048 points over more than 1024 cells, the tile engine's first batch reduces (next to) nothing and the
    # context moves to the sort engine, which merges the 16-byte points directly
    got, exp = _run_cycles(p, cycles, abi.DISP_U16, expect_engine=[TILE, SORT], threads=16)
    assert len(exp) > 1000000
    _close(got, exp)
    _same_cells(got, exp, 0.01)
