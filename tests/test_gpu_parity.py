"""GPU parity: the CUDA path (through the C-ABI, libo3r.so) against the CPU oracle on the same inputs.

Bar (north_star): validity masks, voxel keys, per-voxel counts, colours and output ORDER bit-exact;
coordinates / centroids within 1e-5 relative.  On one GPU the implementation is designed to be
bit-exact for coordinates and centroids too (stable sort + in-order sums), and the tests assert that;
the 1e-5 tolerance is only needed across ranks (tests/test_gpu_multirank.py).
"""
import os

import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi, synth
from online_3d_reconstruction_b200.pose import Pose

pytestmark = pytest.mark.gpu

SMALL = dict(rows=120, cols=200)   # x0 = 25 (unaligned), ROI 155 x 80
SMALL4 = dict(rows=128, cols=256)  # x0 = 32, nx = 204 -> vectorised path


def _frames(seed, n, rows, cols, disp_type=abi.DISP_U8, keep=None, n_kp=0, traj_start=0):
    seq = synth.sequence(seed, n, rows, cols, disp_type=disp_type, traj_start=traj_start)
    rng = np.random.default_rng(seed + 1)
    out = []
    for d, img, T in seq:
        kp = None
        if n_kp:
            kp = np.stack([rng.uniform(-5, cols + 5, n_kp), rng.uniform(-5, rows + 5, n_kp)], 1).astype(np.float32)
        out.append(abi.make_frame(d, img, T, kp_xy=kp, keep=keep))
    return out


def _eq(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    if not np.array_equal(a, b):
        bad = np.nonzero(a.view(np.uint32).reshape(-1, 4) != b.view(np.uint32).reshape(-1, 4))[0]
        raise AssertionError(f"{len(np.unique(bad))} of {len(a)} records differ; first at {bad[0]}: {a[bad[0]]} vs {b[bad[0]]}")


# ---------------------------------------------------------------------------------------------- masks
@pytest.mark.parametrize("J", [1, 3, 15])
@pytest.mark.parametrize("geom", [SMALL, SMALL4])
def test_mask_bit_exact(J, geom):
    keep = []
    p = abi.make_params(jump_pixels=J, **geom)
    fr = _frames(11, 1, geom["rows"], geom["cols"], keep=keep)[0]
    _, mask = ob.create_single_img_pt_cloud(p, fr, abi.DISP_U8, want_mask=True)
    with Pose(p) as P:
        got = P.validityMask(fr)
    assert np.array_equal(got.ravel(), mask)


def test_mask_counts_match_reference_log_720p(real):
    """The reference logged 747674 / 747512 / 747783 valid pixels for frames 1248 / 1249 / 1251
    (--use_segment_labels, jump_pixels 1): labels + per-label plane coefficients evaluated in the kernel."""
    p = abi.make_params(jump_pixels=1, use_segment_labels=True, dont_downsample=True)
    with Pose(p) as P:
        for i in range(3):
            coef, f64 = ob.plane_fit(p, real["labels"][i], real["disp"][i])
            keep = []
            fr = abi.make_frame(None, real["bgr"], np.eye(4), labels=real["labels"][i], plane_coef=coef, keep=keep)
            m = P.validityMask(fr, abi.DISP_F64)
            assert int(m.sum()) == int(real["point_cloud_pts"][i])
            fr64 = abi.make_frame(f64, real["bgr"], np.eye(4), keep=keep)
            pts = P.createAndTransformPtCloud(fr64, abi.DISP_F64)
            exp = ob.create_and_transform_pt_cloud(p, fr64, abi.DISP_F64)
            _eq(pts, exp)
            _eq(P.createAndTransformPtCloud(fr, abi.DISP_F64), exp)


# ----------------------------------------------------------------------------------------------- pre-pass
def test_plane_fit_and_variance_gate_on_real_frames(real):
    """createPlaneFittedDisparityImages + getVariance on the GPU for the three shipped 720p frames: plane coefficients
    bit-identical to the oracle (the normal-equation sums are exact integers), both variances within 1e-10 relative of
    the oracle and equal to what the reference logged (build/output/log.txt:39-42) to its 6 printed digits."""
    p = abi.make_params(jump_pixels=1, use_segment_labels=True)
    with Pose(p) as P:
        for i in range(3):
            labels, disp = real["labels"][i], real["disp"][i]
            coef, f64 = ob.plane_fit(p, labels, disp)
            got_coef, got_var = P.createPlaneFittedDisparityImages(labels, disp)
            assert np.array_equal(got_coef, coef)
            exp_var = ob.get_variance(p, f64, True)
            assert abs(got_var - exp_var) <= 1e-10 * exp_var
            assert f"{got_var:.6g}" == f"{real['plane_fitted_disp_img_var'][i]:.6g}"
            raw_var = P.getVariance(disp)
            assert abs(raw_var - ob.get_variance(p, disp, False)) <= 1e-10 * raw_var
            assert f"{raw_var:.6g}" == f"{real['disp_img_var'][i]:.6g}"


def test_plane_fit_synthetic_labels_small():
    """Ragged cases: a label with no ROI pixel keeps (0,0,0), numbering stops at the first absent label, label 0 is
    never fitted; the coefficients feed straight into the label-mode frame path."""
    rng = np.random.default_rng(5)
    rows, cols = SMALL4["rows"], SMALL4["cols"]
    p = abi.make_params(jump_pixels=1, use_segment_labels=True, **SMALL4)
    labels = np.zeros((rows, cols), np.uint8)
    labels[:, 40:120] = 1
    labels[:60, 120:] = 2
    labels[60:, 120:] = 3
    labels[:10, :30] = 4          # entirely outside the ROI (x < x0, y < bb): fitted as (0, 0, 0)
    labels[70:80, 130:140] = 6    # label 5 is absent: 6 is never reached (pose_functions.cpp:923)
    yy, xx = np.mgrid[:rows, :cols]
    disp = np.clip(90 + 0.05 * xx + 0.1 * yy + rng.normal(0, 1, (rows, cols)), 0, 255).astype(np.uint8)
    coef, f64 = ob.plane_fit(p, labels, disp)
    with Pose(p) as P:
        got_coef, got_var = P.createPlaneFittedDisparityImages(labels, disp)
        assert got_coef.shape == coef.shape == (4, 3)
        assert np.array_equal(got_coef, coef) and not got_coef[3].any()
        exp_var = ob.get_variance(p, f64, True)
        assert abs(got_var - exp_var) <= 1e-10 * max(exp_var, 1e-300)
        keep = []
        bgr = synth.make_frame_images(rng, rows, cols)[1]
        fr = abi.make_frame(None, bgr, np.eye(4), labels=labels, plane_coef=got_coef, keep=keep)
        pts = P.createAndTransformPtCloud(fr, abi.DISP_F64)
    fr64 = abi.make_frame(f64, bgr, np.eye(4), keep=keep)
    _eq(pts, ob.create_and_transform_pt_cloud(p, fr64, abi.DISP_F64))


# ------------------------------------------------------------------------------- points (no downsample)
@pytest.mark.parametrize("J,n_kp", [(1, 0), (1, 50), (7, 300), (0, 1500), (15, 1500)])
@pytest.mark.parametrize("geom", [SMALL, SMALL4])
def test_points_bit_exact_dont_downsample(J, n_kp, geom):
    keep = []
    p = abi.make_params(jump_pixels=J, dont_downsample=True, **geom)
    fr = _frames(5, 1, geom["rows"], geom["cols"], keep=keep, n_kp=n_kp)[0]
    exp = ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)
    with Pose(p) as P:
        got = P.createAndTransformPtCloud(fr)
    _eq(got, exp)


@pytest.mark.parametrize("disp_type", [abi.DISP_U16, abi.DISP_F32, abi.DISP_F64])
@pytest.mark.parametrize("geom", [SMALL, SMALL4])
def test_points_other_disparity_types(disp_type, geom):
    keep = []
    p = abi.make_params(jump_pixels=1, dont_downsample=True, **geom)
    fr = _frames(6, 1, geom["rows"], geom["cols"], disp_type=disp_type, keep=keep)[0]
    exp = ob.create_and_transform_pt_cloud(p, fr, disp_type)
    with Pose(p) as P:
        got = P.createAndTransformPtCloud(fr, disp_type)
    assert len(exp) > 1000
    _eq(got, exp)


def test_points_generic_Q():
    """A Q without the rectified-stereo sparsity takes the generic 4x4 path."""
    keep = []
    Q = list(abi.Q_CAM13)
    Q[1], Q[6], Q[9], Q[12], Q[15] = 1e-3, -2e-3, 5e-4, 1e-5, 0.25
    p = abi.make_params(jump_pixels=1, dont_downsample=True, Q=tuple(Q), **SMALL4)
    fr = _frames(7, 1, SMALL4["rows"], SMALL4["cols"], keep=keep)[0]
    exp = ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)
    with Pose(p) as P:
        got = P.createAndTransformPtCloud(fr)
    _eq(got, exp)


def test_real_frame_720p_dense(real):
    keep = []
    p = abi.make_params(jump_pixels=1, voxel_size=0.05)
    T = synth.trajectory(np.random.default_rng(3), 1)[0]
    fr = abi.make_frame(real["disp"][0], real["bgr"], T, keep=keep)
    exp = ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)
    with Pose(p) as P:
        got = P.createAndTransformPtCloud(fr)
    assert 200000 < len(exp) < 400000
    _eq(got, exp)


def test_empty_frame_and_empty_batch():
    keep = []
    p = abi.make_params(jump_pixels=1, **SMALL)
    fr = abi.make_frame(np.zeros((120, 200), np.uint8), np.zeros((120, 200, 3), np.uint8), np.eye(4), keep=keep)
    with Pose(p) as P:
        assert len(P.createAndTransformPtCloud(fr)) == 0
        assert P.createCycleClouds([fr]).tolist() == [0]
        assert len(P.createCycleClouds([])) == 0
        assert len(P.downsamplePtCloud()) == 0


@pytest.mark.parametrize("sor", [0, 50])
@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_RETAIN])
def test_cycle_with_empty_and_tiny_frames(sor, mode):
    """Ragged cycle: an all-invalid frame, a frame with fewer valid pixels than mean_k + 1, and normal frames — in every
    merge mode, with and without StatisticalOutlierRemoval."""
    keep = []
    geom = SMALL4
    rows, cols = geom["rows"], geom["cols"]
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, sor_mean_k=sor, merge_mode=mode, **geom)
    frames = _frames(190, 4, rows, cols, keep=keep)
    seq = synth.sequence(190, 4, rows, cols)
    empty = abi.make_frame(np.zeros((rows, cols), np.uint8), seq[1][1], seq[1][2], keep=keep)
    tiny_d = np.zeros((rows, cols), np.uint8)
    tiny_d[40:44, 100:107] = 110          # 28 valid pixels
    tiny = abi.make_frame(tiny_d, seq[2][1], seq[2][2], keep=keep)
    cycle = [frames[0], empty, tiny, frames[3]]
    cloud, n, counts = ob.run_cycle(p, cycle, abi.DISP_U8, 2)
    exp = ob.downsample_pt_cloud(p, cloud[:n], True)
    with Pose(p) as P:
        got_counts = P.createCycleClouds(cycle)
        assert np.array_equal(got_counts, counts) and counts[1] == 0 and 0 < counts[2] <= 28
        _eq(P.lastCyclePoints(), cloud[:n])
        got = P.downsamplePtCloud()
    if mode == abi.MERGE_ACCUMULATE_TILED:
        _close(got, exp)
    else:
        _eq(got, exp)


# ------------------------------------------------------------------------------------- per-frame VoxelGrid
@pytest.mark.parametrize("voxel_size", [0.05, 0.1, 0.5])
@pytest.mark.parametrize("geom", [SMALL, SMALL4])
def test_per_frame_voxelgrid_bit_exact(voxel_size, geom):
    keep = []
    p = abi.make_params(jump_pixels=1, voxel_size=voxel_size, **geom)
    fr = _frames(21, 1, geom["rows"], geom["cols"], keep=keep)[0]
    exp = ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)
    with Pose(p) as P:
        got = P.createAndTransformPtCloud(fr)
    assert 0 < len(exp)
    _eq(got, exp)


def test_per_frame_voxelgrid_overflow_passthrough():
    """Leaf so small that dx*dy*dz > INT32_MAX: PCL's guard returns the input unchanged (what config 5's
    voxel_size 0.01 does to a full 4K frame; the small test frame needs a smaller leaf to trip it)."""
    keep = []
    p = abi.make_params(jump_pixels=1, voxel_size=0.002, **SMALL4)
    fr = _frames(22, 1, SMALL4["rows"], SMALL4["cols"], keep=keep)[0]
    p_nd = abi.make_params(jump_pixels=1, voxel_size=0.002, dont_downsample=True, **SMALL4)
    raw = ob.create_and_transform_pt_cloud(p_nd, fr, abi.DISP_U8)
    exp = ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)
    _eq(exp, raw)  # the oracle itself passes through
    with Pose(p) as P:
        got = P.createAndTransformPtCloud(fr)
    _eq(got, exp)


@pytest.mark.parametrize("leaf,min_points", [((0.05, 0.05, 0.05), 0), ((0.3, 0.2, 0.1), 2), ((0.05, 0.05, 1000.0), 3),
                                             ((0.001, 0.001, 0.001), 0)])
def test_voxel_grid_probe_keys_counts_points(leaf, min_points):
    rng = np.random.default_rng(8)
    n = 200000
    pts = np.zeros(n, dtype=abi.POINT)
    pts["x"] = rng.uniform(-8, 12, n).astype(np.float32)
    pts["y"] = rng.uniform(-3, 9, n).astype(np.float32)
    pts["z"] = rng.normal(0, 0.3, n).astype(np.float32)
    pts["rgb"] = rng.integers(0, 1 << 24, n, dtype=np.uint32)
    e_pts, e_keys, e_cnt, e_pass = ob.voxel_grid(pts, leaf, min_points)
    with Pose(abi.make_params(**SMALL)) as P:
        g_pts, g_keys, g_cnt, g_pass = P.voxelGrid(pts, leaf, min_points)
    assert g_pass == e_pass
    assert np.array_equal(g_keys, e_keys)
    assert np.array_equal(g_cnt, e_cnt)
    _eq(g_pts, e_pts)


def test_voxel_grid_reproduces_reference_cloud_ply(golden_dir):
    g = np.load(os.path.join(golden_dir, "cloud_ply.npz"))
    pts = np.zeros(len(g["xyz"]), dtype=abi.POINT)
    pts["x"], pts["y"], pts["z"] = g["xyz"].T
    rgb = g["rgb"].astype(np.uint32)
    pts["rgb"] = (rgb[:, 0] << 16) | (rgb[:, 1] << 8) | rgb[:, 2]
    perm = np.random.default_rng(0).permutation(len(pts))
    for mode in (abi.MERGE_RETAIN, abi.MERGE_ACCUMULATE):
        with Pose(abi.make_params(voxel_size=0.05, min_points_per_voxel=1, merge_mode=mode, **SMALL)) as P:
            P.appendPoints(pts[perm[:30000]])
            P.appendPoints(pts[perm[30000:]])
            _eq(P.downsamplePtCloud(), pts)


# ------------------------------------------------------------------------------------------------- blur
@pytest.mark.parametrize("mode,k", [(abi.BLUR_MEDIAN, 3), (abi.BLUR_MEDIAN, 15), (abi.BLUR_MEDIAN, 31),
                                    (abi.BLUR_BOX, 2), (abi.BLUR_BOX, 5), (abi.BLUR_BOX, 30), (abi.BLUR_BOX, 31),
                                    (abi.BLUR_BILATERAL, 2), (abi.BLUR_BILATERAL, 5), (abi.BLUR_BILATERAL, 30),
                                    (abi.BLUR_BILATERAL, 31), (abi.BLUR_BILATERAL, 101)])
def test_blur_plane_bit_exact(mode, k):
    rng = np.random.default_rng(k)
    src = synth.make_frame_images(rng, 150, 210)[0]
    exp = ob.blur_u8(src, k, mode)
    with Pose(abi.make_params(**SMALL)) as P:
        got = P.blur(src, k, mode)
    assert np.array_equal(got, exp), int((got != exp).sum())


@pytest.mark.parametrize("mode,k", [(abi.BLUR_MEDIAN, 5), (abi.BLUR_MEDIAN, 41), (abi.BLUR_MEDIAN, 127), (abi.BLUR_BOX, 7),
                                    (abi.BLUR_BOX, 127), (abi.BLUR_BILATERAL, 6), (abi.BLUR_BILATERAL, 30)])
def test_blur_plane_full_range_flat_areas_and_odd_width(mode, k):
    """Planes the synthetic disparities do not reach: every 8-bit value incl. 0 and 255 next to large constant areas (the
    sliding median's unchanged-column shortcut, its tracked median jumping across the whole histogram), and an odd width
    (the bilateral kernel's threads own two columns each: the last thread of a row owns one)."""
    rng = np.random.default_rng(1000 + k)
    src = rng.integers(0, 256, (97, 211), dtype=np.uint8)
    src[10:60, 20:120] = 255
    src[30:90, 100:200] = 0
    src[5:25, 150:205] = 77
    exp = ob.blur_u8(src, k, mode)
    with Pose(abi.make_params(**SMALL)) as P:
        got = P.blur(src, k, mode)
    assert np.array_equal(got, exp), int((got != exp).sum())


def test_blur_matches_reference_median_outputs(golden_dir):
    g = np.load(os.path.join(golden_dir, "median_ref.npz"))
    with Pose(abi.make_params(**SMALL)) as P:
        for k in (15, 31):
            assert np.array_equal(P.blur(g["src"], k, abi.BLUR_MEDIAN)[:160, :240], g[f"out{k}"])
            assert np.array_equal(P.blur(g["src_br"], k, abi.BLUR_MEDIAN)[-160:, -240:], g[f"out{k}_br"])


def test_bilateral_on_real_disparity_matches_oracle_and_cv2(golden_dir):
    """The reference's live filter (pose_functions.cpp:1044) on a real 8-bit disparity crop: bit-exact against the
    oracle, and equal to cv2.bilateralFilter at the README's k = 30 (committed fixture)."""
    g = np.load(os.path.join(golden_dir, "bilateral_ref.npz"))
    with Pose(abi.make_params(**SMALL)) as P:
        for k in (5, 30):
            got = P.blur(g["disp"], k, abi.BLUR_BILATERAL)
            assert np.array_equal(got, ob.blur_u8(g["disp"], k, abi.BLUR_BILATERAL))
        assert np.array_equal(got, g["disp_cv2_k30"])   # (k = 5 ties break differently under OpenCV 4.x's FMA)


@pytest.mark.parametrize("mode,k,J", [(abi.BLUR_MEDIAN, 7, 1), (abi.BLUR_BOX, 6, 1), (abi.BLUR_MEDIAN, 5, 4),
                                      (abi.BLUR_BILATERAL, 30, 1), (abi.BLUR_BILATERAL, 9, 3)])
def test_blurred_frame_cloud(mode, k, J):
    keep = []
    p = abi.make_params(jump_pixels=J, voxel_size=0.05, blur_kernel=k, blur_mode=mode, **SMALL4)
    fr = _frames(31, 1, SMALL4["rows"], SMALL4["cols"], keep=keep, n_kp=40)[0]
    exp = ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)
    with Pose(p) as P:
        got = P.createAndTransformPtCloud(fr)
    _eq(got, exp)


def test_blur_rejections():
    keep = []
    p = abi.make_params(jump_pixels=1, blur_kernel=4, blur_mode=abi.BLUR_MEDIAN, **SMALL)
    fr = _frames(1, 1, 120, 200, keep=keep)[0]
    from online_3d_reconstruction_b200.lib import O3RError
    with Pose(p) as P, pytest.raises(O3RError):
        P.createAndTransformPtCloud(fr)  # cv::medianBlur asserts on even ksize -> empty cloud in the reference


# ------------------------------------------------------------------------------------------------- SOR
def _frame_points(seed, geom, J=1, n_kp=0):
    keep = []
    p = abi.make_params(jump_pixels=J, dont_downsample=True, **geom)
    fr = _frames(seed, 1, geom["rows"], geom["cols"], keep=keep, n_kp=n_kp)[0]
    return ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)


@pytest.mark.parametrize("J,n_kp,mean_k", [(1, 0, 50), (3, 200, 50), (7, 400, 20), (15, 1500, 50)])
def test_sor_distances_and_mask_bit_exact(J, n_kp, mean_k):
    """pcl::StatisticalOutlierRemoval (pose_functions.cpp:1673-1686): every point's mean distance to its mean_k nearest
    neighbours must equal the oracle's bit for bit (exact k-NN, float squared distances, ascending double sum), the
    removal mask must be identical; the threshold (cloud statistics, reduced in tree order) within 1e-12 relative."""
    pts = _frame_points(170 + J, SMALL4, J=J, n_kp=n_kp)
    assert len(pts) > mean_k + 1
    keep_o, dist_o = ob.sor(pts, mean_k, 1.0, brute=len(pts) < 6000)
    with Pose(abi.make_params(**SMALL4)) as P:
        keep, dist, thr = P.statisticalOutlierRemoval(pts, mean_k, 1.0)
    assert np.array_equal(dist.view(np.uint32), dist_o.view(np.uint32))
    assert np.array_equal(keep, keep_o)
    d = dist_o.astype(np.float64)
    sq = (dist_o * dist_o).astype(np.float64)
    n = len(d)
    exp_thr = d.sum() / n + np.sqrt((sq.sum() - d.sum() ** 2 / n) / (n - 1))
    assert abs(thr - exp_thr) <= 1e-12 * exp_thr
    assert 0.5 < keep.mean() < 1.0


def test_sor_ragged_clouds():
    """Fewer points than mean_k + 1, duplicates (zero distances), one far outlier, a single point."""
    rng = np.random.default_rng(9)
    base = _frame_points(180, SMALL)[:400].copy()
    with Pose(abi.make_params(**SMALL)) as P:
        for pts in (base[:30], base[:1], np.concatenate([base[:200], base[:200]]), base):
            pts = pts.copy()
            if len(pts) > 100:
                pts["x"][7] += 50.0   # a far outlier: removed
            keep_o, dist_o = ob.sor(pts, 50, 1.0, brute=True)
            keep, dist, _ = P.statisticalOutlierRemoval(pts, 50, 1.0)
            assert np.array_equal(dist.view(np.uint32), dist_o.view(np.uint32))
            assert np.array_equal(keep, keep_o)
            if len(pts) > 100:
                assert keep[7] == 0


@pytest.mark.parametrize("J,n_kp", [(1, 0), (4, 300)])
def test_frame_cloud_with_sor_matches_reference_composition(J, n_kp):
    """createAndTransformPtCloud with the reference's full per-frame downsample (pose_functions.cpp:1654-1709):
    StatisticalOutlierRemoval(50, 1.0), then VoxelGrid(voxel_size / 5) on the filtered cloud."""
    keep = []
    p = abi.make_params(jump_pixels=J, voxel_size=0.05, sor_mean_k=50, **SMALL4)
    frames = _frames(185, 3, SMALL4["rows"], SMALL4["cols"], keep=keep, n_kp=n_kp)
    with Pose(p) as P:
        for fr in frames[:2]:
            _eq(P.createAndTransformPtCloud(fr), ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8))
        cloud, n, counts = ob.run_cycle(p, frames, abi.DISP_U8, 4)
        got_counts = P.createCycleClouds(frames)
        assert np.array_equal(got_counts, counts)
        _eq(P.lastCyclePoints(), cloud[:n])
        _eq(P.downsamplePtCloud(), ob.downsample_pt_cloud(p, cloud[:n], True))
    p0 = abi.make_params(jump_pixels=J, voxel_size=0.05, **SMALL4)
    assert len(ob.create_and_transform_pt_cloud(p0, frames[0], abi.DISP_U8)) > len(ob.create_and_transform_pt_cloud(p, frames[0], abi.DISP_U8))


# ---------------------------------------------------------------------------------- cycles + global cloud
def _oracle_cycles(p, cycles):
    cloud, n = None, 0
    counts = []
    for frames in cycles:
        cloud, n, c = ob.run_cycle(p, frames, abi.DISP_U8, 4, cloud, n)
        counts.append(c)
    big = cloud[:n] if cloud is not None else np.zeros(0, abi.POINT)
    return big, counts


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_RETAIN])
@pytest.mark.parametrize("min_pts", [1, 3])
def test_cycles_merge_equals_one_shot_reference(mode, min_pts):
    """pose.cpp:361-434 over three cycles, then pose.cpp:527-531: the incremental merge must equal the
    reference's single final voxelisation of everything (keys, counts, colours, order AND centroids)."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=min_pts, merge_mode=mode, **geom)
    cycles = [_frames(40, 4, geom["rows"], geom["cols"], keep=keep, traj_start=0),
              _frames(41, 3, geom["rows"], geom["cols"], keep=keep, traj_start=4),
              _frames(42, 4, geom["rows"], geom["cols"], keep=keep, traj_start=5)]
    big, counts = _oracle_cycles(p, cycles)
    exp = ob.downsample_pt_cloud(p, big, True)
    with Pose(p) as P:
        at = 0
        for frames, c in zip(cycles, counts):
            got_c = P.createCycleClouds(frames)
            assert np.array_equal(got_c, c)
            n = int(c.sum())
            _eq(P.lastCyclePoints(), big[at:at + n])
            at += n
        got = P.downsamplePtCloud()
    assert len(exp) > 100
    _eq(got, exp)


def _close(got, exp, rel=1e-5):
    """north_star tolerance for centroids: same records, order, colours (bit-exact) and |dxyz| <= rel * |value| measured
    where the sums live (z + 500: pose_functions.cpp:1666 shifts z before the combined VoxelGrid)."""
    assert got.shape == exp.shape, (got.shape, exp.shape)
    assert np.array_equal(got["rgb"], exp["rgb"])
    for f, shift in (("x", 0.0), ("y", 0.0), ("z", 500.0)):
        a, b = got[f].astype(np.float64) + shift, exp[f].astype(np.float64) + shift
        err = np.abs(a - b)
        lim = rel * np.maximum(np.abs(b), 1e-3)
        assert np.all(err <= lim), f"{f}: max rel err {np.max(err / np.maximum(np.abs(b), 1e-3)):.3g}"


@pytest.mark.parametrize("min_pts", [1, 2, 5])
@pytest.mark.parametrize("voxel", [0.05, 0.2])
def test_tiled_merge_keys_counts_colours_exact_centroids_1e5(min_pts, voxel):
    """O3R_MERGE_ACCUMULATE_TILED: tile partial sums are merged instead of single items.  The set of cells (keys), their
    order, the per-cell point counts (probed through min_points_per_voxel = 1, 2, 5) and the colour sums must equal
    the one-shot reference voxelisation exactly; centroids within 1e-5 relative (float reassociation)."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=voxel, min_points_per_voxel=min_pts,
                        merge_mode=abi.MERGE_ACCUMULATE_TILED, **geom)
    cycles = [_frames(140, 4, geom["rows"], geom["cols"], keep=keep, traj_start=0),
              _frames(141, 3, geom["rows"], geom["cols"], keep=keep, traj_start=4),
              _frames(142, 4, geom["rows"], geom["cols"], keep=keep, traj_start=5)]
    big, counts = _oracle_cycles(p, cycles)
    exp = ob.downsample_pt_cloud(p, big, True)
    with Pose(p) as P:
        at = 0
        for frames, c in zip(cycles, counts):
            assert np.array_equal(P.createCycleClouds(frames), c)
            n = int(c.sum())
            _eq(P.lastCyclePoints(), big[at:at + n])   # the per-frame clouds themselves stay bit-exact
            at += n
        got = P.downsamplePtCloud()
    assert len(exp) > 50
    _close(got, exp)
    # cell keys of the outputs: identical sequence
    inv = np.float32(1.0) / np.float32(voxel)
    for f in ("x", "y"):
        assert np.array_equal(np.floor(got[f] * inv), np.floor(exp[f] * inv))


def test_tiled_merge_is_reproducible_and_matches_exact_mode_cells():
    """Two runs of the tiled mode give identical bits (no atomics on floats, fixed fold order); the exact-order mode on
    the same input has the same cells, counts and colours."""
    keep = []
    geom = SMALL4
    frames = _frames(150, 5, geom["rows"], geom["cols"], keep=keep, n_kp=0)
    outs = []
    for mode in (abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE):
        p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=mode, **geom)
        with Pose(p) as P:
            P.createCycleClouds(frames[:3])
            P.createCycleClouds(frames[3:])
            outs.append(P.downsamplePtCloud())
    _eq(outs[0], outs[1])
    _close(outs[0], outs[2])


def test_tiled_merge_full_resolution_720p_against_exact_mode():
    """Full-size property: at 1280x720 (748 000 points per frame, tiles that straddle frames and partial last tiles)
    the tiled mode and the exact-order mode agree on cells, counts (min_points 3) and colours, centroids 1e-5."""
    keep = []
    frames = _frames(160, 3, 720, 1280, keep=keep)
    outs = []
    for mode in (abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE):
        p = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=3, merge_mode=mode)
        with Pose(p) as P:
            P.createCycleClouds(frames[:2])
            P.createCycleClouds(frames[2:])
            outs.append(P.downsamplePtCloud())
    assert len(outs[1]) > 10000
    _close(outs[0], outs[1])


def test_downsample_device_result_matches_host_result():
    torch = pytest.importorskip("torch")
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, **geom)
    with Pose(p) as P:
        P.createCycleClouds(_frames(45, 3, geom["rows"], geom["cols"], keep=keep))
        host = P.downsamplePtCloud()
        ptr, n = P.downsamplePtCloudDevice()
        assert n == len(host)
        class DevArr:   # wrap the raw device pointer for torch
            __cuda_array_interface__ = {"shape": (n * 16,), "typestr": "|u1", "data": (ptr, False), "version": 2}
        buf = torch.as_tensor(DevArr(), device="cuda").cpu().numpy().view(abi.POINT)
        _eq(buf, host)


def test_dont_downsample_cycle_returns_cloud_big():
    keep = []
    p = abi.make_params(jump_pixels=2, dont_downsample=True, **SMALL)
    cycles = [_frames(50, 3, 120, 200, keep=keep), _frames(51, 2, 120, 200, keep=keep, traj_start=3)]
    big, _ = _oracle_cycles(p, cycles)
    with Pose(p) as P:
        for frames in cycles:
            P.createCycleClouds(frames)
        assert P.cloudSize() == len(big)
        _eq(P.downsamplePtCloud(), big)


def test_retain_mode_icp_retro_transform():
    """pose.cpp:350-354: cloud_big is re-transformed by tf_icp every cycle before the new frames are appended."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.1, merge_mode=abi.MERGE_RETAIN, **geom)
    cycles = [_frames(60, 3, geom["rows"], geom["cols"], keep=keep), _frames(61, 3, geom["rows"], geom["cols"], keep=keep, traj_start=3)]
    tf = np.eye(4, dtype=np.float32)
    c, s = np.float32(np.cos(0.01)), np.float32(np.sin(0.01))
    tf[0, 0], tf[0, 1], tf[1, 0], tf[1, 1] = c, -s, s, c
    tf[:3, 3] = [0.03, -0.02, 0.01]
    cloud, n, _ = ob.run_cycle(p, cycles[0], abi.DISP_U8, 4)
    cloud[:n] = ob.transform_pt_cloud(cloud[:n], tf)
    cloud, n, _ = ob.run_cycle(p, cycles[1], abi.DISP_U8, 4, cloud, n)
    exp = ob.downsample_pt_cloud(p, cloud[:n], True)
    with Pose(p) as P:
        P.createCycleClouds(cycles[0])
        P.transformPtCloud(tf)
        P.createCycleClouds(cycles[1])
        _eq(P.downsamplePtCloud(), exp)
    from online_3d_reconstruction_b200.lib import O3RError
    with Pose(abi.make_params(jump_pixels=1, **geom)) as P, pytest.raises(O3RError):
        P.transformPtCloud(tf)  # accumulate mode cannot re-bin


def test_prefetch_is_transparent():
    """o3r_frames_prefetch only moves the H2D copies earlier (double-buffered staging): same results; a prefetch of
    other frames is ignored; buffers may be reused for the cycle after next."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=3, voxel_size=0.05, **geom)
    cycles = [_frames(90 + c, 3, geom["rows"], geom["cols"], keep=keep, n_kp=20, traj_start=3 * c) for c in range(4)]
    with Pose(p) as A, Pose(p) as B:
        for c in cycles:
            A.createCycleClouds(c)
        arrs = [(abi.Frame * len(c))(*c) for c in cycles]
        B.prefetchCycle(arrs[0])
        for i, arr in enumerate(arrs):
            if i + 1 < len(arrs):
                B.prefetchCycle(arrs[i + 1] if i != 1 else arrs[0])   # cycle 2's prefetch is a wrong guess: ignored
            B.createCycleClouds(arr)
            _eq(B.lastCyclePoints(), A.lastCyclePoints()) if i == len(arrs) - 1 else None
        _eq(A.downsamplePtCloud(), B.downsamplePtCloud())


def test_device_pointer_entry_point_matches_host_entry_point():
    torch = pytest.importorskip("torch")
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, **geom)
    seq = synth.sequence(70, 3, geom["rows"], geom["cols"])
    host = [abi.make_frame(d, img, T, keep=keep) for d, img, T in seq]
    dev = []
    for d, img, T in seq:
        td, ti = torch.from_numpy(d).cuda(), torch.from_numpy(img).cuda()
        keep.extend([td, ti])
        f = abi.Frame()
        f.disp, f.disp_step = td.data_ptr(), d.strides[0]
        f.bgr, f.bgr_step = ti.data_ptr(), img.strides[0]
        f.T = host[len(dev)].T
        dev.append(f)
    torch.cuda.synchronize()
    with Pose(p) as A, Pose(p) as B:
        ca = A.createCycleClouds(host)
        cb = B.createCycleClouds(dev, device_pointers=True)
        assert np.array_equal(ca, cb)
        _eq(A.downsamplePtCloud(), B.downsamplePtCloud())


# ------------------------------------------------------------------------- full-size properties (720p)
def test_full_resolution_properties_720p():
    """BASELINE configs[1] geometry (1280x720, jump_pixels 1, voxel_size 0.05), 8 frames in two cycles — too big for
    the oracle to be quick, so size-independent properties are checked instead:
      * the incremental merge (engine 2, ACCUMULATE) and the one-shot PCL-style voxelisation of the retained cloud
        (engine 1, RETAIN) are independent code paths and must agree bit for bit,
      * the combined cloud is strictly increasing in its (y-cell, x-cell) key with one point per cell,
      * per-frame counts are consistent with the batch, and re-voxelising the result returns it unchanged."""
    keep = []
    frames = _frames(1002, 8, 720, 1280, keep=keep)
    p_acc = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=1, merge_mode=abi.MERGE_ACCUMULATE)
    p_ret = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=1, merge_mode=abi.MERGE_RETAIN)
    with Pose(p_acc) as A, Pose(p_ret) as R:
        ca = np.concatenate([A.createCycleClouds(frames[:5]), A.createCycleClouds(frames[5:])])
        cr = np.concatenate([R.createCycleClouds(frames[:5]), R.createCycleClouds(frames[5:])])
        assert np.array_equal(ca, cr) and np.all(ca > 300000) and np.all(ca <= 748000)
        assert R.cloudSize() == int(cr.sum())
        a, r = A.downsamplePtCloud(), R.downsamplePtCloud()
        _eq(a, r)
        assert A.cloudSize() == len(a) > 10000
        # strictly increasing cell keys
        sh = a.copy()
        sh["z"] += np.float32(500)
        inv = np.float32(1.0) / np.float32(0.05)
        i = np.floor(sh["x"] * inv).astype(np.int64)
        j = np.floor(sh["y"] * inv).astype(np.int64)
        key = (j << 21) + i
        assert np.all(np.diff(key) > 0)
        # idempotence through the stand-alone probe (same leaf, same z shift)
        again, _, counts, passthrough = A.voxelGrid(sh, (0.05, 0.05, 1000.0), 1)
        assert not passthrough and np.all(counts == 1)
        _eq(again, sh)

