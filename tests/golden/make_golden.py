"""Generates tests/golden/*.npz from the reference's shipped artefacts (run in the build container,
where /root/reference exists; the GPU box only sees the committed .npz files).

    python tests/golden/make_golden.py

Sources (relative to /root/reference/build):
  disparities/{1248,1249,1251}.png, segmentlabels/{same}.png  real 1280x720 frames (no colour plane)
  output/log.txt:39-46,64          valid-pixel counts + variances the reference logged for them
  images/1248.png                  input of the median / bilateral crops below
  output/medianBlurred_{15,31}.png cv::medianBlur outputs of images/1248.png written by the reference
  output/bilateralFiltered_{15,31}.png cv::bilateralFilter(img, k, 2k, k/2) outputs written by the reference
  cloud.ply                        a combined-grid VoxelGrid output of the reference (voxel_size 0.05)
plus one fixture that comes from OpenCV (cv2 4.13 of the build container) rather than from the reference's files:
  reproject_cv2.npz                cv2.gemm(Q, [x y d 1]^T) for a generic Q over a small frame's scan ROI
  planefit_cv2.npz                 per-label plane coefficients of the three real frames computed the reference's way with
                                   cv2.gemm / cv2.invert(DECOMP_SVD)
Decoding PNGs needs cv2 (present in the build container only).
"""
import os

import cv2
import numpy as np

R = "/root/reference/build/"
OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    # --- real frames + the numbers the reference logged for them (log.txt) ---
    nums = [1248, 1249, 1251]
    disp = np.stack([cv2.imread(R + f"disparities/{n}.png", cv2.IMREAD_GRAYSCALE) for n in nums])
    labels = np.stack([cv2.imread(R + f"segmentlabels/{n}.png", cv2.IMREAD_GRAYSCALE) for n in nums])
    # no colour plane: the logged numbers depend on disparities and labels only, and a 720p photo alone would put the file
    # over 1 MB (the tests draw a seeded synthetic colour plane instead)
    np.savez_compressed(
        os.path.join(OUT, "real_frames.npz"), img_nums=np.array(nums), disp=disp, labels=labels,
        # log.txt:39,40,42 "index i disp_img_var V plane_fitted_disp_img_var P"; :45,46,64 "point_clout_pts"
        disp_img_var=np.array([2.27913, 2.64813, 2.08488]),
        plane_fitted_disp_img_var=np.array([1.63692, 1.49152, 1.64115]),
        point_cloud_pts=np.array([747674, 747512, 747783]))
    # --- median blur: crops of the reference's own outputs (top-left corner: exercises the border) ---
    img = cv2.imread(R + "images/1248.png")
    m15 = cv2.imread(R + "output/medianBlurred_15.png")
    m31 = cv2.imread(R + "output/medianBlurred_31.png")
    np.savez_compressed(os.path.join(OUT, "median_ref.npz"),
                        src=img[:200, :280, 1].copy(),          # green channel, input crop incl. halo
                        out15=m15[:160, :240, 1].copy(), out31=m31[:160, :240, 1].copy(),
                        src_br=img[-200:, -280:, 2].copy(),     # bottom-right corner, red channel
                        out15_br=m15[-160:, -240:, 2].copy(), out31_br=m31[-160:, -240:, 2].copy())
    # --- bilateral filter: crops of the reference's own outputs (cv::bilateralFilter(img, k, 2k, k/2), 3 channels),
    #     and a cn = 1 case (a real disparity crop) filtered by this container's cv2 (the reference call, pose_functions.cpp:1044)
    b15 = cv2.imread(R + "output/bilateralFiltered_15.png")
    b31 = cv2.imread(R + "output/bilateralFiltered_31.png")
    d1248 = cv2.imread(R + "disparities/1248.png", cv2.IMREAD_GRAYSCALE)
    dcrop = d1248[300:460, 500:740].copy()
    np.savez_compressed(os.path.join(OUT, "bilateral_ref.npz"),
                        src=img[:200, :280].copy(),             # BGR input crop (top-left corner: border + halo)
                        out15=b15[:160, :240].copy(), out31=b31[:160, :240].copy(),
                        disp=dcrop, disp_cv2_k5=cv2.bilateralFilter(dcrop, 5, 10, 2),
                        disp_cv2_k30=cv2.bilateralFilter(dcrop, 30, 60, 15), cv2_version=np.array(cv2.__version__))
    # --- cloud.ply vertices ---
    raw = open(R + "cloud.ply", "rb").read()
    h = raw.index(b"end_header\n") + len(b"end_header\n")
    n = 55940
    v = np.frombuffer(raw[h:h + 15 * n], dtype=np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"),
                                                         ("r", "u1"), ("g", "u1"), ("b", "u1")]))
    np.savez_compressed(os.path.join(OUT, "cloud_ply.npz"), header=np.frombuffer(raw[:h], dtype=np.uint8),
                        xyz=np.stack([v["x"], v["y"], v["z"]], 1), rgb=np.stack([v["r"], v["g"], v["b"]], 1),
                        trailer=np.frombuffer(raw[h + 15 * n:], dtype=np.uint8))
    # --- the reprojection's matrix product through OpenCV itself: cv::Mat_<double>(4x4) * (4x1) = cv::gemm, for a GENERIC Q
    #     (every entry non-zero: with the rectified-stereo Q at most two terms per row are non-zero and any summation order
    #     gives the same bits).  Pins the oracle's left-to-right row sums (pose_functions.cpp:1074, :1111) on OpenCV 4.x.
    rng = np.random.default_rng(77)
    rows, cols, bb = 60, 100, 20
    x0 = cols // 8
    Qg = rng.normal(size=(4, 4)) * np.array([1.0, 1.0, 1.0, 100.0])
    Qg[3] = [1e-4, -2e-4, 1.7, 0.3]          # keeps the homogeneous coordinate away from 0
    dimg = rng.integers(65, 128, (rows, cols)).astype(np.uint8)
    ys, xs = np.mgrid[bb:rows - bb, x0:cols - bb]
    vecs = np.stack([xs.ravel(), ys.ravel(), dimg[ys.ravel(), xs.ravel()], np.ones(xs.size)], 1).astype(np.float64)
    prod = np.stack([cv2.gemm(Qg, v.reshape(4, 1).copy(), 1.0, None, 0.0).ravel() for v in vecs])
    np.savez_compressed(os.path.join(OUT, "reproject_cv2.npz"), Q=Qg, disp=dimg, gemm=prod, cv2_version=np.array(cv2.__version__))
    # --- the plane fit the way the reference writes it (pose_functions.cpp:940-965), through OpenCV: A (N x 3), At * A by cv::gemm,
    #     cv::invert(DECOMP_SVD), (AtAinv * At) * b — the oracle solves the same normal equations from exact integer sums with its
    #     own 3 x 3 inverse, so its coefficients differ from these in the last digits (tests bound the difference and its effect)
    rows, cols, bb = 720, 1280, 20
    x0 = cols // 8
    coefs = np.zeros((3, 8, 3))
    n_planes = []
    for i in range(3):
        cc = []
        for cl in range(1, 1024):
            ys, xs = np.nonzero(labels[i] == cl)
            if len(xs) == 0:
                break
            m = (xs > x0) & (xs < cols - bb) & (ys > bb) & (ys < rows - bb)
            A = np.stack([xs[m].astype(np.float64), ys[m].astype(np.float64), np.ones(int(m.sum()))], 1)
            b = disp[i][ys[m], xs[m]].astype(np.float64).reshape(-1, 1)
            At = np.ascontiguousarray(A.T)
            _, inv = cv2.invert(cv2.gemm(At, A, 1.0, None, 0.0), flags=cv2.DECOMP_SVD)
            cc.append(cv2.gemm(cv2.gemm(inv, At, 1.0, None, 0.0), b, 1.0, None, 0.0).ravel())
        coefs[i, :len(cc)] = np.array(cc)
        n_planes.append(len(cc))
    np.savez_compressed(os.path.join(OUT, "planefit_cv2.npz"), coef=coefs, n_planes=np.array(n_planes), cv2_version=np.array(cv2.__version__))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
