"""ctypes mirror of include/o3r.h (struct layouts, enums, numpy record dtypes).

Pure declarations: no library is loaded here, so the checker's binding in tests/ can share the
struct definitions while the product never touches the checker.
"""
import ctypes as C

import numpy as np

O3R_OK = 0
O3R_ERR_INVALID = -1
O3R_ERR_CUDA = -2
O3R_ERR_CAPACITY = -3
O3R_ERR_UNSUPPORTED = -4
O3R_ERR_NOMEM = -5

DISP_U8, DISP_U16, DISP_F32, DISP_F64 = 0, 1, 2, 3
BLUR_MEDIAN, BLUR_BOX, BLUR_BILATERAL = 0, 1, 2
MERGE_ACCUMULATE, MERGE_RETAIN, MERGE_ACCUMULATE_TILED, MERGE_ACCUMULATE_FUSED = 0, 1, 2, 3

DISP_NP = {DISP_U8: np.uint8, DISP_U16: np.uint16, DISP_F32: np.float32, DISP_F64: np.float64}

#: o3r_point — 16-byte XYZRGB record (pcl::PointXYZRGB payload, SURVEY §8a row P)
POINT = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("rgb", "<u4")])
#: o3r_cell — 40-byte partial-sum record exchanged between ranks
CELL = np.dtype([("key", "<u8"), ("sx", "<f4"), ("sy", "<f4"), ("sz", "<f4"), ("n", "<u4"),
                 ("sr", "<u4"), ("sg", "<u4"), ("sb", "<u4"), ("pad", "<u4")])
assert POINT.itemsize == 16 and CELL.itemsize == 40


class Params(C.Structure):
    """o3r_params: the `Pose` members the path reads (pose.h:93-98,108,118,126-128,149,168)."""
    _fields_ = [
        ("rows", C.c_int), ("cols", C.c_int),
        ("cols_start_aft_cutout", C.c_int),
        ("bounding_box", C.c_int),
        ("min_disparity", C.c_double),
        ("Q", C.c_double * 16),
        ("jump_pixels", C.c_int),
        ("blur_kernel", C.c_int),
        ("blur_mode", C.c_int),
        ("voxel_size", C.c_double),
        ("min_points_per_voxel", C.c_uint),
        ("dont_downsample", C.c_int),
        ("use_segment_labels", C.c_int),
        ("disp_divisor", C.c_double),
        ("merge_mode", C.c_int),
        ("device", C.c_int),
        ("max_batch_frames", C.c_int),
        ("sor_mean_k", C.c_int),
        ("sor_stddev_mul", C.c_double),
    ]


class Frame(C.Structure):
    """o3r_frame: one accepted image's inputs (pose.cpp:596-607, pose_functions.cpp:1035-1051)."""
    _fields_ = [
        ("disp", C.c_void_p), ("disp_step", C.c_size_t),
        ("bgr", C.c_void_p), ("bgr_step", C.c_size_t),
        ("labels", C.c_void_p), ("labels_step", C.c_size_t),
        ("plane_coef", C.c_void_p), ("n_planes", C.c_int),
        ("kp_xy", C.c_void_p), ("n_kp", C.c_int),
        ("T", C.c_float * 16),
    ]


#: Q loaded by the reference (pose.h:127 -> build/data_files/cam13calib.yml, matrix Q)
Q_CAM13 = (1.0, 0.0, 0.0, -5.2425751876831055e+02,
           0.0, 1.0, 0.0, -5.1381009292602539e+02,
           0.0, 0.0, 0.0, 4.2300101518980237e+03,
           0.0, 0.0, 1.6853548938735339e+00, 0.0)


class RegisterParams(C.Structure):
    """o3r_register_params: Gauss-Newton limits of o3r_cloud_register."""
    _fields_ = [
        ("max_iterations", C.c_int),
        ("max_distance", C.c_double),
        ("min_rotation", C.c_double),
        ("min_translation", C.c_double),
        ("degenerate_ratio", C.c_double),
    ]


class RegisterStats(C.Structure):
    """o3r_register_stats: what o3r_cloud_register reports besides T_out."""
    _fields_ = [
        ("iterations", C.c_uint32), ("converged", C.c_uint32), ("rank", C.c_uint32),
        ("n_inliers", C.c_uint32),
        ("rms_initial", C.c_double), ("rms_final", C.c_double),
        ("pivot", C.c_double * 3),
        ("info", C.c_double * 36),
    ]


def make_register_params(voxel_size, *, max_iterations=20, max_distance=None, min_rotation=1e-5, min_translation=1e-4,
                         degenerate_ratio=1e-3):
    """The library's defaults (max_distance = 3 * voxel_size)."""
    r = RegisterParams()
    r.max_iterations = max_iterations
    r.max_distance = 3.0 * voxel_size if max_distance is None else max_distance
    r.min_rotation, r.min_translation, r.degenerate_ratio = min_rotation, min_translation, degenerate_ratio
    return r


def make_params(rows=720, cols=1280, *, jump_pixels=10, voxel_size=0.1, min_points_per_voxel=1,
                blur_kernel=1, blur_mode=BLUR_MEDIAN, dont_downsample=False, use_segment_labels=False,
                Q=Q_CAM13, min_disparity=64.0, bounding_box=20, cutout_ratio=8, disp_divisor=200.0,
                merge_mode=MERGE_ACCUMULATE, device=0, max_batch_frames=64, sor_mean_k=0, sor_stddev_mul=1.0):
    """Defaults are the reference's (pose.h:93-98,108,118,126,149,168)."""
    p = Params()
    p.rows, p.cols = rows, cols
    p.cols_start_aft_cutout = cols // cutout_ratio  # pose_functions.cpp:638
    p.bounding_box = bounding_box
    p.min_disparity = min_disparity
    p.Q = (C.c_double * 16)(*Q)
    p.jump_pixels = jump_pixels
    p.blur_kernel = blur_kernel
    p.blur_mode = blur_mode
    p.voxel_size = voxel_size
    p.min_points_per_voxel = min_points_per_voxel
    p.dont_downsample = int(dont_downsample)
    p.use_segment_labels = int(use_segment_labels)
    p.disp_divisor = disp_divisor
    p.merge_mode = merge_mode
    p.device = device
    p.max_batch_frames = max_batch_frames
    p.sor_mean_k = sor_mean_k          # the reference: 50 whenever jump_pixels > 0 (pose_functions.cpp:1673-1686)
    p.sor_stddev_mul = sor_stddev_mul
    return p


def scan_dims(p):
    """(ny, nx) of the grid scan (pose_functions.cpp:1094-1128); (0, 0) when jump_pixels == 0."""
    J = p.jump_pixels
    if J <= 0:
        return 0, 0
    ny = max(0, (p.rows - 2 * p.bounding_box + J - 1) // J)
    nx = max(0, (p.cols - p.bounding_box - p.cols_start_aft_cutout + J - 1) // J)
    return ny, nx


def _ptr(a):
    return None if a is None else a.ctypes.data


def make_frame(disp, bgr, T, *, labels=None, plane_coef=None, kp_xy=None, keep=None):
    """Builds an o3r_frame over numpy arrays (host).  `keep` (a list) receives references that must
    outlive the struct."""
    f = Frame()
    disp = np.ascontiguousarray(disp) if disp is not None else None
    bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
    if disp is not None:
        f.disp, f.disp_step = _ptr(disp), disp.strides[0]
    f.bgr, f.bgr_step = _ptr(bgr), bgr.strides[0]
    if labels is not None:
        labels = np.ascontiguousarray(labels, dtype=np.uint8)
        f.labels, f.labels_step = _ptr(labels), labels.strides[0]
    if plane_coef is not None:
        plane_coef = np.ascontiguousarray(plane_coef, dtype=np.float64).reshape(-1, 3)
        f.plane_coef, f.n_planes = _ptr(plane_coef), plane_coef.shape[0]
    if kp_xy is not None:
        kp_xy = np.ascontiguousarray(kp_xy, dtype=np.float32).reshape(-1, 2)
        f.kp_xy, f.n_kp = _ptr(kp_xy), kp_xy.shape[0]
    f.T = (C.c_float * 16)(*np.asarray(T, dtype=np.float32).reshape(16))
    if keep is not None:
        keep.extend([disp, bgr, labels, plane_coef, kp_xy])
    return f
