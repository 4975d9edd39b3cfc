"""Host-side mirror of the reference's `Pose` hot-path interface over the C-ABI (include/o3r.h).

Method names follow the reference so the parity tests read like the reference's own call sites:

    createAndTransformPtCloud   pose.cpp:596-636
    createCycleClouds           pose.cpp:361-434   (the 7-thread fan-out + ordered concat + append)
    transformPtCloud            pose.cpp:350-354   (cloud_big <- tf_icp * cloud_big)
    downsamplePtCloud           pose_functions.cpp:1654-1709 (combinedPtCloud = true)

Everything computes on the GPU through libo3r.so; numpy only carries buffers across the boundary.
"""
import ctypes as C

import numpy as np

from . import abi, lib


class Pose:
    """One reconstruction context (= the read-only `Pose` state after populateData + the global cloud)."""

    world, rank = 1, 0   # the communicator this context is part of (commInit); 1, 0 without one

    def __init__(self, params=None, **kw):
        self._L = lib.load()
        self.params = params if params is not None else abi.make_params(**kw)
        h = C.c_void_p()
        rc = self._L.o3r_create(C.byref(self.params), C.byref(h))
        if rc != 0:
            raise lib.O3RError(rc, self._L.o3r_last_error(None).decode())
        self._h = h

    # -- plumbing ------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.o3r_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise lib.O3RError(rc, self._L.o3r_last_error(self._h).decode())

    @property
    def handle(self):
        return self._h

    @property
    def max_points_per_frame(self):
        ny, nx = abi.scan_dims(self.params)
        return ny * nx

    def lastCyclePartials(self):
        return int(self._L.o3r_last_batch_partials(self._h))

    def launch_count(self):
        return int(self._L.o3r_launch_count(self._h))

    def stream(self):
        return self._L.o3r_stream(self._h)

    def sync(self):
        self._check(self._L.o3r_sync(self._h))

    def profile(self, enable):
        """Per-kernel CUDA-event timing on/off (clears the records)."""
        self._check(self._L.o3r_profile(self._h, int(enable)))

    def profileRead(self):
        """-> {kernel name: (launches, total_ms)} since profile(True)."""
        buf = C.create_string_buffer(1 << 16)
        self._check(self._L.o3r_profile_read(self._h, buf, len(buf)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, ms = line.split("\t")
            out[name.strip("()")] = (int(n), float(ms))
        return out

    # -- per-frame path --------------------------------------------------------------------------------
    def createAndTransformPtCloud(self, frame, disp_type=abi.DISP_U8):
        """pose.cpp:596-636 for one accepted image -> structured array of abi.POINT."""
        cap = max(1, self.max_points_per_frame + (frame.n_kp if self.params.jump_pixels != 1 else 0))
        out = np.empty(cap, dtype=abi.POINT)
        n = C.c_size_t(0)
        self._check(self._L.o3r_frame_cloud(self._h, C.byref(frame), disp_type, out.ctypes.data, cap, C.byref(n)))
        return out[:n.value].copy()

    def validityMask(self, frame, disp_type=abi.DISP_U8):
        """The `disp > minDisparity` mask of the grid scan (pose_functions.cpp:1094-1107), row-major (ny, nx)."""
        ny, nx = abi.scan_dims(self.params)
        mask = np.zeros(max(1, ny * nx), dtype=np.uint8)
        n = C.c_size_t(0)
        self._check(self._L.o3r_frame_mask(self._h, C.byref(frame), disp_type, mask.ctypes.data, mask.size, C.byref(n)))
        return mask[:n.value].reshape(ny, nx)

    def createCycleClouds(self, frames, disp_type=abi.DISP_U8, device_pointers=False):
        """pose.cpp:361-434: all accepted frames of a cycle, concatenated in order and appended to the
        global cloud.  Returns the per-frame point counts.  An empty list is a cycle without frames (n = 0): on a sharded
        RETAIN context it is how a rank with no frame in the cycle keeps step with the others."""
        n = len(frames)
        arr = frames if isinstance(frames, C.Array) else (abi.Frame * n)(*frames)
        counts = np.zeros(max(n, 1), dtype=np.uint32)
        fn = self._L.o3r_frames_cloud_dev if device_pointers else self._L.o3r_frames_cloud
        self._check(fn(self._h, arr, n, disp_type, counts.ctypes.data))
        return counts[:n]

    def prefetchCycle(self, frames, disp_type=abi.DISP_U8):
        """Starts the host->device copies of the NEXT cycle's frames (pass the same array to createCycleClouds later)."""
        n = len(frames)
        arr = frames if isinstance(frames, C.Array) else (abi.Frame * n)(*frames)
        self._check(self._L.o3r_frames_prefetch(self._h, arr, n, disp_type))
        return arr

    def cancelPrefetch(self):
        """Drops announced prefetches; afterwards the library no longer references their host buffers."""
        self._check(self._L.o3r_frames_prefetch_cancel(self._h))

    def lastCyclePoints(self):
        n = C.c_size_t(0)
        self._check(self._L.o3r_last_batch_points(self._h, None, 0, C.byref(n)))
        out = np.empty(max(1, n.value), dtype=abi.POINT)
        self._check(self._L.o3r_last_batch_points(self._h, out.ctypes.data, out.size, C.byref(n)))
        return out[:n.value]

    def lastCycleEngine(self):
        """Engine of the last cycle: 2 = the fused tile engine, 1 = the fused bucket engine, 0 = the sort engine."""
        return int(self._L.o3r_last_batch_engine(self._h))

    def setKeepFrameVoxels(self, keep):
        """Parity probe of MERGE_ACCUMULATE_FUSED: lastCyclePoints() then returns the per-frame voxel centroids of the
        cycle as a multiset (no particular order)."""
        self._check(self._L.o3r_set_keep_frame_voxels(self._h, int(keep)))

    # -- global cloud ------------------------------------------------------------------------------------
    def transformPtCloud(self, T):
        """pose.cpp:353 transformPtCloud(cloud_big, cloud_big, tf_icp) — RETAIN mode only."""
        Tc = (C.c_float * 16)(*np.asarray(T, dtype=np.float32).reshape(16))
        self._check(self._L.o3r_cloud_transform(self._h, Tc))

    def appendPoints(self, pts):
        pts = np.ascontiguousarray(pts, dtype=abi.POINT)
        self._check(self._L.o3r_cloud_append(self._h, pts.ctypes.data, pts.size))

    def cloudSize(self):
        n = C.c_size_t(0)
        self._check(self._L.o3r_cloud_size(self._h, C.byref(n)))
        return n.value

    def clearCloud(self):
        self._check(self._L.o3r_cloud_clear(self._h))

    def downsamplePtCloud(self, out=None):
        """pose_functions.cpp:1654-1709 with combinedPtCloud = true on the global cloud (pose.cpp:530).

        On a sharded RETAIN context this is a collective: every rank returns the combined-grid cells it owns
        (exchange.owner_of), in ascending voxel index; the union ordered by cell key is the single-GPU output bit for bit.
        On a pass-through grid and with dont_downsample every rank returns its own points.  The result is kept until the
        local cloud changes, so the size query and the fill below communicate once."""
        n = C.c_size_t(0)
        if out is None:
            self._check(self._L.o3r_cloud_downsample(self._h, None, 0, C.byref(n)))
            out = np.empty(max(1, n.value), dtype=abi.POINT)
        self._check(self._L.o3r_cloud_downsample(self._h, out.ctypes.data, out.size, C.byref(n)))
        return out[:n.value]

    def downsamplePtCloudDevice(self):
        """Same as downsamplePtCloud but the result stays in device memory -> (device pointer, n records)."""
        ptr, n = C.c_void_p(), C.c_size_t(0)
        self._check(self._L.o3r_cloud_downsample_dev(self._h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def trackCloudChanges(self, enable=True):
        """Change tracking of the resident cloud (accumulate modes) on / off.  Enabling (or re-enabling) makes the next
        cloudChanges() return the full state; disabling frees the tracking buffers."""
        self._check(self._L.o3r_cloud_track_changes(self._h, int(enable)))

    def cloudChanges(self):
        """The cells whose point count grew since the last call (every cell after trackCloudChanges), count >=
        min_points_per_voxel, ascending cell key -> (points, keys u64, counts u32).  Upserting them by key into a
        key-sorted map keeps it equal to downsamplePtCloud(), bit for bit.  Consumes the changes."""
        n = C.c_size_t(0)
        self._check(self._L.o3r_cloud_changes(self._h, None, None, None, 0, C.byref(n)))
        cap = max(1, n.value)
        out = np.empty(cap, dtype=abi.POINT)
        keys = np.empty(cap, dtype=np.uint64)
        counts = np.empty(cap, dtype=np.uint32)
        self._check(self._L.o3r_cloud_changes(self._h, out.ctypes.data, keys.ctypes.data, counts.ctypes.data, cap,
                                              C.byref(n)))
        k = n.value
        return out[:k], keys[:k], counts[:k]

    def cloudChangesDevice(self):
        """Same as cloudChanges but the records stay in device memory owned by the context (valid until the next call on
        it) -> (points pointer, keys pointer, counts pointer, n).  Consumes the changes."""
        pts, keys, counts, n = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_size_t(0)
        self._check(self._L.o3r_cloud_changes_dev(self._h, C.byref(pts), C.byref(keys), C.byref(counts), C.byref(n)))
        return pts.value, keys.value, counts.value, n.value

    def exportCells(self):
        """Every resident cell (accumulate modes), ascending key, cells below min_points_per_voxel included: a bit copy of
        the accumulators as an abi.CELL array.  With a communicator: the shard this rank owns."""
        n = C.c_size_t(0)
        self._check(self._L.o3r_cloud_export_cells(self._h, None, 0, C.byref(n)))
        out = np.empty(max(1, n.value), dtype=abi.CELL)
        self._check(self._L.o3r_cloud_export_cells(self._h, out.ctypes.data, out.size, C.byref(n)))
        return out[:n.value]

    def importCells(self, cells):
        """Merges abi.CELL records into the resident map as one cycle (sums added in input order after the resident ones).
        All or nothing: a refused record raises O3RError (O3R_ERR_INVALID) naming its index, and nothing is merged."""
        cells = np.ascontiguousarray(cells, dtype=abi.CELL)
        self._check(self._L.o3r_cloud_import_cells(self._h, cells.ctypes.data, cells.size))

    def exportPoints(self):
        """cloud_big in order, exactly (MERGE_RETAIN or dont_downsample, no communicator); appendPoints is the import."""
        n = C.c_size_t(0)
        self._check(self._L.o3r_cloud_export_points(self._h, None, 0, C.byref(n)))
        out = np.empty(max(1, n.value), dtype=abi.POINT)
        self._check(self._L.o3r_cloud_export_points(self._h, out.ctypes.data, out.size, C.byref(n)))
        return out[:n.value]

    def registerCloud(self, pts, T_init=None, device_pointer=None, **params):
        """o3r_cloud_register: the rigid T (starting from T_init, identity by default) such that T * p lies on the resident
        map (accumulate modes) -> (T_out float32 4x4, stats dict).  params: max_iterations, max_distance, min_rotation,
        min_translation, degenerate_ratio (abi.make_register_params defaults).  device_pointer=(ptr, n) registers device
        points through o3r_cloud_register_dev instead of the host array `pts`."""
        rp = abi.make_register_params(self.params.voxel_size, **params)
        T0 = np.eye(4, dtype=np.float32) if T_init is None else np.asarray(T_init, dtype=np.float32).reshape(4, 4)
        Tin = (C.c_float * 16)(*T0.reshape(16))
        Tout = (C.c_float * 16)()
        st = abi.RegisterStats()
        if device_pointer is not None:
            ptr, n = device_pointer
            self._check(self._L.o3r_cloud_register_dev(self._h, ptr, n, Tin, C.byref(rp), Tout, C.byref(st)))
        else:
            pts = np.ascontiguousarray(pts, dtype=abi.POINT)
            self._check(self._L.o3r_cloud_register(self._h, pts.ctypes.data, pts.size, Tin, C.byref(rp), Tout, C.byref(st)))
        stats = dict(iterations=st.iterations, converged=st.converged, rank=st.rank, n_inliers=st.n_inliers,
                     rms_initial=st.rms_initial, rms_final=st.rms_final, pivot=np.array(st.pivot[:]),
                     info=np.array(st.info[:]).reshape(6, 6))
        return np.array(Tout[:], dtype=np.float32).reshape(4, 4), stats

    def meshCloud(self, max_step=float("inf")):
        """o3r_cloud_mesh: the resident map's height field as triangles (accumulate modes) -> (vertices as abi.POINT,
        exactly downsamplePtCloud(); normals (n, 3) float32, (0, 0, 0) where no plane fits; triangles (m, 3) uint32
        vertex indices, counter-clockwise seen from above).  A triangle is kept iff its largest |dz| is <= max_step."""
        nv, nt = C.c_size_t(0), C.c_size_t(0)
        self._check(self._L.o3r_cloud_mesh(self._h, float(max_step), None, None, 0, C.byref(nv), None, 0, C.byref(nt)))
        verts = np.empty(max(1, nv.value), dtype=abi.POINT)
        normals = np.empty((max(1, nv.value), 3), dtype=np.float32)
        tris = np.empty((max(1, nt.value), 3), dtype=np.uint32)
        self._check(self._L.o3r_cloud_mesh(self._h, float(max_step), verts.ctypes.data, normals.ctypes.data, nv.value,
                                           C.byref(nv), tris.ctypes.data, nt.value, C.byref(nt)))
        return verts[:nv.value], normals[:nv.value], tris[:nt.value]

    def meshCloudDevice(self, max_step=float("inf")):
        """Same as meshCloud but the result stays in device memory owned by the context (valid until the next call on it)
        -> (vertices pointer, normals pointer, n vertices, triangles pointer, n triangles)."""
        v, nrm, t = C.c_void_p(), C.c_void_p(), C.c_void_p()
        nv, nt = C.c_size_t(0), C.c_size_t(0)
        self._check(self._L.o3r_cloud_mesh_dev(self._h, float(max_step), C.byref(v), C.byref(nrm), C.byref(nv), C.byref(t),
                                               C.byref(nt)))
        return v.value, nrm.value, nv.value, t.value, nt.value

    # -- stand-alone stages --------------------------------------------------------------------------------
    def voxelGrid(self, pts, leaf, min_points=0):
        """pcl::VoxelGrid on a host cloud -> (points, keys u64, counts u32, passthrough)."""
        pts = np.ascontiguousarray(pts, dtype=abi.POINT)
        n = pts.size
        out = np.empty(max(1, n), dtype=abi.POINT)
        keys = np.empty(max(1, n), dtype=np.uint64)
        counts = np.empty(max(1, n), dtype=np.uint32)
        m, pt = C.c_size_t(0), C.c_int(0)
        lx, ly, lz = (np.float32(v) for v in leaf)
        self._check(self._L.o3r_voxel_grid(self._h, pts.ctypes.data, n, lx, ly, lz, min_points, out.ctypes.data,
                                           out.size, C.byref(m), keys.ctypes.data, counts.ctypes.data, C.byref(pt)))
        k = m.value
        return out[:k].copy(), keys[:k].copy(), counts[:k].copy(), bool(pt.value)

    def statisticalOutlierRemoval(self, pts, mean_k=50, stddev_mul=1.0):
        """pcl::StatisticalOutlierRemoval on a host cloud -> (keep mask u8, mean neighbour distances f32, threshold)."""
        pts = np.ascontiguousarray(pts, dtype=abi.POINT)
        keep = np.zeros(max(1, pts.size), dtype=np.uint8)
        dist = np.zeros(max(1, pts.size), dtype=np.float32)
        thr = C.c_double(0)
        self._check(self._L.o3r_sor(self._h, pts.ctypes.data, pts.size, mean_k, float(stddev_mul), keep.ctypes.data,
                                    dist.ctypes.data, C.byref(thr)))
        return keep[:pts.size], dist[:pts.size], thr.value

    def blur(self, src, kernel, mode):
        src = np.ascontiguousarray(src, dtype=np.uint8)
        dst = np.empty_like(src)
        self._check(self._L.o3r_blur_u8(self._h, src.ctypes.data, src.strides[0], src.shape[0], src.shape[1], kernel,
                                        mode, dst.ctypes.data, dst.strides[0]))
        return dst

    # -- pre-pass ------------------------------------------------------------------------------------------
    def getVariance(self, disp):
        """pose_functions.cpp:1007-1028 getVariance(disp_img, false): the bad-frame gate's statistic (pose.cpp:187)."""
        disp = np.ascontiguousarray(disp, dtype=np.uint8)
        v = C.c_double(0)
        self._check(self._L.o3r_disp_variance(self._h, disp.ctypes.data, disp.strides[0], C.byref(v)))
        return v.value

    def createPlaneFittedDisparityImages(self, labels, disp):
        """pose_functions.cpp:900-985 -> (plane coefficients [n_planes, 3] f64, plane_fitted_disp_img_var)."""
        labels = np.ascontiguousarray(labels, dtype=np.uint8)
        disp = np.ascontiguousarray(disp, dtype=np.uint8)
        coef = np.zeros((255, 3), dtype=np.float64)
        n, v = C.c_int(0), C.c_double(0)
        self._check(self._L.o3r_plane_fit(self._h, labels.ctypes.data, labels.strides[0], disp.ctypes.data, disp.strides[0],
                                          coef.ctypes.data, 255, C.byref(n), C.byref(v)))
        return coef[:n.value].copy(), v.value

    # -- multi-GPU exchange inside the library (NCCL bound at run time): see include/o3r.h ----------------------
    @staticmethod
    def commUniqueId():
        """rank 0: the 128-byte NCCL id every rank passes to commInit (send it over any host channel)."""
        buf = C.create_string_buffer(128)
        rc = lib.load().o3r_comm_unique_id(buf)
        if rc != 0:
            raise lib.O3RError(rc, lib.load().o3r_last_error(None).decode())
        return buf.raw

    def commInit(self, world, rank, uid, slot_cells):
        """Collective: attaches a communicator of `world` ranks.  Accumulate modes: the cycle's cells are exchanged by
        exchangeCycle into fixed slots of `slot_cells` cells.  RETAIN (or dont_downsample): the cloud must still be empty;
        each rank keeps the points of its frames (f mod world == rank), slot_cells is not used, and downsamplePtCloud
        becomes the collective.  All ranks make the same sequence of createCycleClouds / transformPtCloud / clearCloud calls."""
        self._check(self._L.o3r_comm_init(self._h, world, rank, C.c_char_p(uid), slot_cells))
        self.world, self.rank = world, rank

    def commDestroy(self):
        self._check(self._L.o3r_comm_destroy(self._h))
        self.world, self.rank = 1, 0

    def exchangeCycle(self):
        """Collective, asynchronous: partial cells of the last cycle -> owners (grouped ncclSend/ncclRecv) -> merge.
        On a sharded RETAIN context it is a no-op (the points stay where they were made), so one driver loop serves every
        mode."""
        self._check(self._L.o3r_exchange_cycle(self._h))
