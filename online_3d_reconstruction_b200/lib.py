"""Loads libo3r.so (the C-ABI library built from csrc/) and declares every entry point of include/o3r.h.

There is no fallback: if the shared library is missing or a CUDA device is absent the calls fail loudly.
"""
import ctypes as C
import os

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libo3r.so")

#: every symbol include/o3r.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "o3r_create", "o3r_destroy", "o3r_last_error", "o3r_version", "o3r_host_alloc", "o3r_host_free",
    "o3r_frame_cloud", "o3r_frames_cloud", "o3r_frames_cloud_dev", "o3r_frames_prefetch", "o3r_frames_prefetch_cancel", "o3r_last_batch_points",
    "o3r_cloud_transform", "o3r_cloud_append", "o3r_cloud_downsample", "o3r_cloud_downsample_dev", "o3r_cloud_size",
    "o3r_cloud_clear", "o3r_cloud_track_changes", "o3r_cloud_changes", "o3r_cloud_changes_dev",
    "o3r_cloud_export_cells", "o3r_cloud_import_cells", "o3r_cloud_export_points",
    "o3r_voxel_grid", "o3r_blur_u8", "o3r_frame_mask", "o3r_disp_variance", "o3r_plane_fit", "o3r_sor", "o3r_last_batch_partials",
    "o3r_set_keep_frame_voxels", "o3r_last_batch_engine",
    "o3r_comm_unique_id", "o3r_comm_init", "o3r_comm_attach", "o3r_comm_destroy", "o3r_exchange_cycle",
    "o3r_launch_count", "o3r_stream", "o3r_sync", "o3r_profile", "o3r_profile_read",
]

_lib = None


class O3RError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"o3r error {code}: {msg}")
        self.code = code


def load():
    """Returns the ctypes handle of libo3r.so with argtypes set.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(
            f"{SO_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C online_3d_reconstruction_b200/csrc).  There is no CPU fallback.")
    L = C.CDLL(SO_PATH)
    vp, sz, szp = C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)
    P, F = C.POINTER(abi.Params), C.POINTER(abi.Frame)
    L.o3r_create.argtypes = [P, C.POINTER(vp)]
    L.o3r_destroy.argtypes = [vp]
    L.o3r_destroy.restype = None
    L.o3r_last_error.argtypes = [vp]
    L.o3r_last_error.restype = C.c_char_p
    L.o3r_host_alloc.argtypes = [sz]
    L.o3r_host_alloc.restype = vp
    L.o3r_host_free.argtypes = [vp]
    L.o3r_host_free.restype = None
    L.o3r_frame_cloud.argtypes = [vp, F, C.c_int, vp, sz, szp]
    L.o3r_frames_cloud.argtypes = [vp, F, C.c_int, C.c_int, vp]
    L.o3r_frames_cloud_dev.argtypes = [vp, F, C.c_int, C.c_int, vp]
    L.o3r_frames_prefetch.argtypes = [vp, F, C.c_int, C.c_int]
    L.o3r_frames_prefetch_cancel.argtypes = [vp]
    L.o3r_last_batch_points.argtypes = [vp, vp, sz, szp]
    L.o3r_cloud_transform.argtypes = [vp, C.POINTER(C.c_float)]
    L.o3r_cloud_append.argtypes = [vp, vp, sz]
    L.o3r_cloud_downsample.argtypes = [vp, vp, sz, szp]
    L.o3r_cloud_downsample_dev.argtypes = [vp, C.POINTER(vp), szp]
    L.o3r_cloud_size.argtypes = [vp, szp]
    L.o3r_cloud_clear.argtypes = [vp]
    L.o3r_cloud_track_changes.argtypes = [vp, C.c_int]
    L.o3r_cloud_changes.argtypes = [vp, vp, vp, vp, sz, szp]
    L.o3r_cloud_changes_dev.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), szp]
    L.o3r_cloud_export_cells.argtypes = [vp, vp, sz, szp]
    L.o3r_cloud_import_cells.argtypes = [vp, vp, sz]
    L.o3r_cloud_export_points.argtypes = [vp, vp, sz, szp]
    L.o3r_voxel_grid.argtypes = [vp, vp, sz, C.c_float, C.c_float, C.c_float, C.c_uint, vp, sz, szp, vp, vp,
                                 C.POINTER(C.c_int)]
    L.o3r_blur_u8.argtypes = [vp, vp, sz, C.c_int, C.c_int, C.c_int, C.c_int, vp, sz]
    L.o3r_frame_mask.argtypes = [vp, F, C.c_int, vp, sz, szp]
    L.o3r_last_batch_partials.argtypes = [vp]
    L.o3r_last_batch_partials.restype = C.c_size_t
    L.o3r_sor.argtypes = [vp, vp, sz, C.c_int, C.c_double, vp, vp, C.POINTER(C.c_double)]
    L.o3r_disp_variance.argtypes = [vp, vp, sz, C.POINTER(C.c_double)]
    L.o3r_plane_fit.argtypes = [vp, vp, sz, vp, sz, vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double)]
    L.o3r_set_keep_frame_voxels.argtypes = [vp, C.c_int]
    L.o3r_last_batch_engine.argtypes = [vp]
    L.o3r_comm_unique_id.argtypes = [vp]
    L.o3r_comm_init.argtypes = [vp, C.c_int, C.c_int, vp, sz]
    L.o3r_comm_attach.argtypes = [vp, vp, C.c_int, C.c_int, sz]
    L.o3r_comm_destroy.argtypes = [vp]
    L.o3r_exchange_cycle.argtypes = [vp]
    L.o3r_launch_count.argtypes = [vp]
    L.o3r_launch_count.restype = C.c_uint64
    L.o3r_stream.argtypes = [vp]
    L.o3r_stream.restype = vp
    L.o3r_sync.argtypes = [vp]
    L.o3r_profile.argtypes = [vp, C.c_int]
    L.o3r_profile_read.argtypes = [vp, C.c_char_p, sz]
    _lib = L
    return L
