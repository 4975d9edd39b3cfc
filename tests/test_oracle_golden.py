"""Pins the CPU oracle against the artefacts the reference ships (SURVEY §4 / §8c).

The reference has no tests; these are its de-facto golden vectors (tests/golden/make_golden.py).
"""
import os

import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi


def test_disp_variance_matches_reference_log(real):
    """getVariance on raw u8 disparity == build/output/log.txt:39-42 (6 significant figures)."""
    p = abi.make_params(jump_pixels=1)
    for i in range(3):
        v = ob.get_variance(p, real["disp"][i], False)
        assert f"{v:.6g}" == f"{real['disp_img_var'][i]:.6g}"


def test_plane_fit_variance_and_mask_count_match_reference_log(real):
    """createPlaneFittedDisparityImages + getVariance(planeFitted) and the valid-pixel count of
    createSingleImgPtCloud (jump_pixels=1, --use_segment_labels) == log.txt:39-46,64."""
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, use_segment_labels=True)
    bgr = real["bgr"]
    for i in range(3):
        coef, f64 = ob.plane_fit(p, real["labels"][i], real["disp"][i])
        v = ob.get_variance(p, f64, True)
        assert f"{v:.6g}" == f"{real['plane_fitted_disp_img_var'][i]:.6g}"
        keep = []
        fr = abi.make_frame(f64, bgr, np.eye(4), keep=keep)
        pts, mask = ob.create_single_img_pt_cloud(p, fr, abi.DISP_F64, want_mask=True)
        assert len(pts) == int(real["point_cloud_pts"][i]) == int(mask.sum())
        # labels + per-label (a,b,c) evaluated in place is the same image
        fr2 = abi.make_frame(None, bgr, np.eye(4), labels=real["labels"][i], plane_coef=coef, keep=keep)
        pts2 = ob.create_single_img_pt_cloud(p, fr2, abi.DISP_F64)
        assert np.array_equal(pts, pts2)


def test_plane_fit_against_opencv_gemm_and_svd_inverse(real, golden_dir):
    """The reference fits each label's plane as (invert(At*A, DECOMP_SVD) * At) * b over the N x 3 design matrix
    (pose_functions.cpp:940-965).  The fixture holds those coefficients computed with cv2 4.13 on the three shipped frames; the
    oracle (exact integer normal equations + its own 3 x 3 inverse) must agree to 1e-9 relative, give the same validity mask
    (the reference's logged point counts) and the same cloud except for a handful of coordinates that round the other way
    (<= 1 ulp, <= 3 per 2.2 M): that is how far the label-mode cloud can sit from the true binary's."""
    g = np.load(os.path.join(golden_dir, "planefit_cv2.npz"))
    p = abi.make_params(jump_pixels=1, use_segment_labels=True, dont_downsample=True)
    for i in range(3):
        n = int(g["n_planes"][i])
        cv = g["coef"][i, :n]
        coef, _ = ob.plane_fit(p, real["labels"][i], real["disp"][i])
        coef = np.asarray(coef).reshape(-1, 3)
        assert coef.shape == cv.shape
        assert np.max(np.abs(coef - cv) / np.abs(cv)) < 1e-9
        keep = []
        fa = abi.make_frame(None, real["bgr"], np.eye(4), labels=real["labels"][i], plane_coef=coef, keep=keep)
        fb = abi.make_frame(None, real["bgr"], np.eye(4), labels=real["labels"][i], plane_coef=cv, keep=keep)
        pa = ob.create_single_img_pt_cloud(p, fa, abi.DISP_F64)
        pb = ob.create_single_img_pt_cloud(p, fb, abi.DISP_F64)
        assert len(pa) == len(pb) == int(real["point_cloud_pts"][i])
        assert np.array_equal(pa["rgb"], pb["rgb"])
        differing = 0
        for f in ("x", "y", "z"):
            ulps = np.abs(pa[f].view(np.int32).astype(np.int64) - pb[f].view(np.int32))
            assert ulps.max() <= 1
            differing += int((ulps != 0).sum())
        assert differing <= 3, differing


def test_median_matches_reference_outputs(golden_dir):
    """cv::medianBlur(images/1248.png, 15|31) as written by the reference (output/medianBlurred_*.png)."""
    g = np.load(os.path.join(golden_dir, "median_ref.npz"))
    for k in (15, 31):
        out = ob.blur_u8(g["src"], k, abi.BLUR_MEDIAN)
        assert np.array_equal(out[:160, :240], g[f"out{k}"])
        out = ob.blur_u8(g["src_br"], k, abi.BLUR_MEDIAN)
        assert np.array_equal(out[-160:, -240:], g[f"out{k}_br"])


def test_bilateral_matches_reference_outputs(golden_dir):
    """cv::bilateralFilter(images/1248.png, k, 2k, k/2) as written by the reference (output/bilateralFiltered_{15,31}.png,
    OpenCV 3.1).  The restatement reproduces them up to +-1 LSB on < 1e-4 of the samples (OpenCV 4.13 in the build
    container differs from the 3.1 artefacts by the same amount, SURVEY section 4); k/2 must be the INTEGER division."""
    g = np.load(os.path.join(golden_dir, "bilateral_ref.npz"))
    for k in (15, 31):
        out = ob.bilateral_u8(g["src"], k, 2 * k, k // 2)[:160, :240]
        d = out.astype(int) - g[f"out{k}"].astype(int)
        assert np.abs(d).max() <= 1
        assert np.mean(d != 0) < 1e-4
    wrong = ob.bilateral_u8(g["src"], 15, 30, 7.5)[:160, :240]      # float division: clearly off
    assert np.mean(wrong != g["out15"]) > 1e-3


def test_bilateral_single_channel_matches_cv2(golden_dir):
    """The path's own case (u8 disparity, cn = 1) against cv2.bilateralFilter 4.13 run in the build container on a real
    disparity crop, for the reference's parameterisation (k, 2k, k/2).  k = 30 (the README's value) agrees on every
    pixel.  At k = 5 the window mean of an 8-bit disparity image sits on an exact .5 tie for a quarter of the pixels, and
    OpenCV 4.x accumulates with fused multiply-adds where 3.1 (the reference, SSE mul + add) and this restatement do
    not, so ties break differently: only |difference| <= 1 is asserted there."""
    g = np.load(os.path.join(golden_dir, "bilateral_ref.npz"))
    out = ob.blur_u8(g["disp"], 30, abi.BLUR_BILATERAL)
    assert np.array_equal(out, g["disp_cv2_k30"])
    d = ob.blur_u8(g["disp"], 5, abi.BLUR_BILATERAL).astype(int) - g["disp_cv2_k5"].astype(int)
    assert np.abs(d).max() <= 1


def test_median_rejects_even_kernel():
    src = np.zeros((8, 8), np.uint8)
    with pytest.raises(RuntimeError):
        ob.blur_u8(src, 4, abi.BLUR_MEDIAN)


def test_box_small_cases():
    """cv::blur model: anchor k/2, BORDER_REFLECT_101, round-half-even."""
    src = np.arange(25, dtype=np.uint8).reshape(5, 5) * 10
    out = ob.blur_u8(src, 3, abi.BLUR_BOX)
    pad = np.pad(src.astype(np.int64), 1, mode="reflect")
    S = sum(pad[dy:dy + 5, dx:dx + 5] for dy in range(3) for dx in range(3))
    q, r = np.divmod(S, 9)
    exp = q + (2 * r > 9)
    assert np.array_equal(out, exp.astype(np.uint8))
    # even kernel: window [x-1, x] for k=2, ties go to even
    src = np.array([[0, 1, 0, 1]] * 2, dtype=np.uint8)
    out = ob.blur_u8(src, 2, abi.BLUR_BOX)
    # sums: reflect101 of col -1 is col 1 -> S = 2*(src[x-1]+src[x]); x=0: 2*(1+0)=2 -> 0.5 -> 0
    assert out.tolist() == [[0, 0, 0, 0]] * 2


def _ply_points(golden_dir):
    g = np.load(os.path.join(golden_dir, "cloud_ply.npz"))
    pts = np.zeros(len(g["xyz"]), dtype=abi.POINT)
    pts["x"], pts["y"], pts["z"] = g["xyz"].T
    rgb = g["rgb"].astype(np.uint32)
    pts["rgb"] = (rgb[:, 0] << 16) | (rgb[:, 1] << 8) | rgb[:, 2]
    return pts


def test_combined_voxelgrid_reproduces_reference_cloud_ply(golden_dir):
    """build/cloud.ply is a combined-grid VoxelGrid output (voxel_size 0.05): one point per XY cell in
    ascending (j, i) order with every z on the float(+500, -500) lattice.  Re-voxelising it — in the
    original or any shuffled order — must return it bit-exactly (order, cell function, z round trip)."""
    pts = _ply_points(golden_dir)
    p = abi.make_params(voxel_size=0.05, min_points_per_voxel=1)
    out = ob.downsample_pt_cloud(p, pts, True)
    assert np.array_equal(out, pts)
    perm = np.random.default_rng(0).permutation(len(pts))
    assert np.array_equal(ob.downsample_pt_cloud(p, pts[perm], True), pts)
    # keys strictly increasing in the shipped order
    sh = pts.copy()
    sh["z"] += np.float32(500)
    _, keys, counts, pt = ob.voxel_grid(sh, (0.05, 0.05, 1000.0), 1)
    assert not pt and np.all(np.diff(keys.astype(np.int64)) > 0) and np.all(counts == 1)


def test_min_points_per_voxel(golden_dir):
    pts = _ply_points(golden_dir)[:2000]
    dup = np.concatenate([pts, pts[::2]])
    p = abi.make_params(voxel_size=0.05, min_points_per_voxel=2)
    out = ob.downsample_pt_cloud(p, dup, True)
    assert np.array_equal(out, pts[::2])


def test_author_known_answer_frame():
    """build/disparities/pointCloud.m:36-48: disparity 128 everywhere, 142 in rows 99..199 x cols 199..399;
    image green, red in the block.  Z = Q23 / (Q32 * d)."""
    disp = np.full((720, 1280), 128, np.uint8)
    disp[99:200, 199:400] = 142
    bgr = np.zeros((720, 1280, 3), np.uint8)
    bgr[:, :, 1] = 255
    bgr[99:200, 199:400, 1] = 0
    bgr[99:200, 199:400, 2] = 255
    p = abi.make_params(jump_pixels=1, dont_downsample=True)
    keep = []
    pts = ob.create_single_img_pt_cloud(p, abi.make_frame(disp, bgr, np.eye(4), keep=keep), abi.DISP_U8)
    assert len(pts) == 748000
    f, a = abi.Q_CAM13[11], abi.Q_CAM13[14]
    z = pts["z"].reshape(680, 1100)
    assert np.all(z[100 - 20:200 - 20, 200 - 160:400 - 160] == np.float32(f / (a * 142)))
    assert z[0, 0] == np.float32(f / (a * 128)) and abs(float(z[0, 0]) - 19.608) < 1e-3
    rgb = pts["rgb"].reshape(680, 1100)
    assert rgb[0, 0] == 0x00FF00 and rgb[100, 100] == 0xFF0000
    # first scanned pixel is (x0=160, y=20)
    assert pts["x"][0] == np.float32((160 + abi.Q_CAM13[3]) * (1.0 / (a * 128)))


def test_generic_q_row_sums_match_cv_gemm(golden_dir):
    """cv::Mat_<double> Q * vec (pose_functions.cpp:1074, :1111) is cv::gemm.  For a Q with sixteen non-zero entries the order of
    the four products' sum matters in the last bit; the fixture holds cv2.gemm's own results (OpenCV 4.13, make_golden.py) for
    every scan pixel of a small frame, and the oracle's points must equal (float)(v_i * (1.0 / v_3)) of exactly those doubles."""
    g = np.load(os.path.join(golden_dir, "reproject_cv2.npz"))
    rows, cols = g["disp"].shape
    p = abi.make_params(rows=rows, cols=cols, jump_pixels=1, dont_downsample=True, Q=tuple(g["Q"].ravel()))
    keep = []
    fr = abi.make_frame(g["disp"], np.zeros((rows, cols, 3), np.uint8), np.eye(4), keep=keep)
    pts = ob.create_single_img_pt_cloud(p, fr, abi.DISP_U8)
    v = g["gemm"]
    assert len(pts) == len(v)
    r = 1.0 / v[:, 3]
    for i, f in enumerate(("x", "y", "z")):
        assert np.array_equal(pts[f], (v[:, i] * r).astype(np.float32)), f
    # and the same products summed pairwise (what a two-accumulator gemm would do) do NOT reproduce them: the pin is not vacuous
    q = g["Q"]
    ys, xs = np.mgrid[20:rows - 20, cols // 8:cols - 20]
    vec = np.stack([xs.ravel(), ys.ravel(), g["disp"][ys.ravel(), xs.ravel()], np.ones(xs.size)], 1).astype(np.float64)
    a = q[None, :, :] * vec[:, None, :]
    pair = (a[:, :, 0] + a[:, :, 2]) + (a[:, :, 1] + a[:, :, 3])
    assert (pair != v).any()


def test_voxelgrid_overflow_guard_passthrough():
    """PCL: dx*dy*dz > INT32_MAX -> 'Leaf size is too small', output = input."""
    rng = np.random.default_rng(1)
    pts = np.zeros(1000, dtype=abi.POINT)
    pts["x"], pts["y"], pts["z"] = (rng.uniform(0, 10, (3, 1000))).astype(np.float32)
    out, keys, counts, passthrough = ob.voxel_grid(pts, (0.002, 0.002, 0.002), 0)
    assert passthrough and np.array_equal(out, pts) and np.all(counts == 1)
    out, _, counts, passthrough = ob.voxel_grid(pts, (0.5, 0.5, 0.5), 0)
    assert not passthrough and counts.sum() == 1000 and len(out) < 1000


def test_empty_inputs():
    pts = np.zeros(0, dtype=abi.POINT)
    out, keys, counts, pt = ob.voxel_grid(pts, (0.1, 0.1, 0.1), 0)
    assert len(out) == 0 and not pt
    p = abi.make_params(jump_pixels=1, dont_downsample=True)
    keep = []
    fr = abi.make_frame(np.zeros((720, 1280), np.uint8), np.zeros((720, 1280, 3), np.uint8), np.eye(4), keep=keep)
    assert len(ob.create_and_transform_pt_cloud(p, fr, abi.DISP_U8)) == 0


def test_generate_tmat_structure():
    """generateTmat (pose_functions.cpp:1178-1356): identity attitude -> known closed form; bad norm throws."""
    T = ob.generate_tmat(1.0, 2.0, 3.0, 0.0, 0.0, 0.0, 1.0)
    assert T[3].tolist() == [0, 0, 0, 1]
    R = T[:3, :3].astype(np.float64)
    assert np.allclose(R @ R.T, np.eye(3), atol=1e-6) and abs(abs(np.linalg.det(R)) - 1) < 1e-6
    # camera looks down: image z (depth) maps to world -z
    assert T[2, 2] < -0.99
    with pytest.raises(ValueError):
        ob.generate_tmat(0, 0, 0, 0.5, 0.5, 0.5, 0.9)
    # float product is left-to-right row*col accumulation
    a = np.random.default_rng(0).normal(size=(4, 4)).astype(np.float32)
    b = np.random.default_rng(1).normal(size=(4, 4)).astype(np.float32)
    m = ob.mat4_mul(a, b)
    exp = np.zeros((4, 4), np.float32)
    for i in range(4):
        for j in range(4):
            s = np.float32(a[i, 0] * b[0, j])
            for k in range(1, 4):
                s = np.float32(s + np.float32(a[i, k] * b[k, j]))
            exp[i, j] = s
    assert np.array_equal(m, exp)


# ------------------------------------------------------------------------------ StatisticalOutlierRemoval
def _sor_numpy(pts, mean_k, mul):
    """Independent restatement in numpy (all pairs): float squared distances, double sqrt, ascending sum."""
    xyz = np.stack([pts["x"], pts["y"], pts["z"]], 1).astype(np.float32)
    n = len(xyz)
    dist = np.zeros(n, np.float32)
    for i in range(n):
        d = xyz[i] - xyz                                      # float32
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        nn = np.sort(d2)[:mean_k + 1]
        s = 0.0
        for v in nn[1:]:
            s += np.sqrt(np.float64(v))
        dist[i] = np.float32(s / mean_k)
    s, sq = 0.0, 0.0
    for v in dist:
        s += float(v)
        sq += float(np.float32(v * v))
    mean = s / n
    thr = mean + mul * np.sqrt((sq - s * s / n) / (n - 1))
    return (~(dist.astype(np.float64) > thr)).astype(np.uint8), dist


def test_sor_known_answer_line_of_points():
    """Points on a line at unit spacing plus one far point: with mean_k = 2 the inner points' mean neighbour distance
    is 1, the ends' 1.5, the outlier's is large and it alone is removed."""
    pts = np.zeros(8, dtype=abi.POINT)
    pts["x"][:7] = np.arange(7)
    pts["x"][7] = 100.0
    keep, dist = ob.sor(pts, 2, 1.0, brute=True)
    assert dist[:7].tolist() == [1.5, 1.0, 1.0, 1.0, 1.0, 1.0, 1.5]
    assert dist[7] == np.float32((94.0 + 95.0) / 2)
    assert keep.tolist() == [1] * 7 + [0]


def test_sor_grid_search_equals_all_pairs_and_numpy():
    """The oracle's grid k-NN is exact: identical to its own all-pairs search and to an independent numpy restatement
    (surface-like cloud with outliers, duplicates and a cloud smaller than mean_k + 1)."""
    rng = np.random.default_rng(11)
    n = 1500
    pts = np.zeros(n, dtype=abi.POINT)
    pts["x"], pts["y"] = rng.uniform(0, 3, n).astype(np.float32), rng.uniform(0, 2, n).astype(np.float32)
    pts["z"] = (0.05 * np.round(rng.normal(0, 1, n)) + 0.01 * pts["x"]).astype(np.float32)   # layered, tilted
    pts["z"][:20] += rng.uniform(1, 5, 20).astype(np.float32)                                  # outliers
    pts[100:120] = pts[200:220]                                                                # duplicates
    for cloud, k in ((pts, 50), (pts, 7), (pts[:40], 50), (pts[:1], 50)):
        kb, db = ob.sor(cloud, k, 1.0, brute=True)
        kg, dg = ob.sor(cloud, k, 1.0, brute=False, threads=3)
        assert np.array_equal(db.view(np.uint32), dg.view(np.uint32)) and np.array_equal(kb, kg)
    kn, dn = _sor_numpy(pts[:400], 10, 1.0)
    ko, do = ob.sor(pts[:400], 10, 1.0, brute=False)
    assert np.array_equal(dn.view(np.uint32), do.view(np.uint32)) and np.array_equal(kn, ko)
    assert ko[:20].sum() < 5   # the lifted points are (mostly) removed


def test_downsample_applies_sor_only_per_frame_and_only_for_jump_pixels():
    """pose_functions.cpp:1673: SOR runs iff !combinedPtCloud && jump_pixels > 0."""
    rng = np.random.default_rng(12)
    n = 3000
    pts = np.zeros(n, dtype=abi.POINT)
    pts["x"], pts["y"] = rng.uniform(0, 1, n).astype(np.float32), rng.uniform(0, 1, n).astype(np.float32)
    pts["z"][:30] = 3.0
    on = abi.make_params(jump_pixels=1, voxel_size=0.05, sor_mean_k=50, rows=64, cols=64)
    off = abi.make_params(jump_pixels=1, voxel_size=0.05, sor_mean_k=0, rows=64, cols=64)
    kp_only = abi.make_params(jump_pixels=0, voxel_size=0.05, sor_mean_k=50, rows=64, cols=64)
    a, b, c = (ob.downsample_pt_cloud(p, pts, False) for p in (on, off, kp_only))
    assert len(a) < len(b) and np.array_equal(b, c)
    assert np.array_equal(ob.downsample_pt_cloud(on, pts, True), ob.downsample_pt_cloud(off, pts, True))
