/*
 * o3r.h — C ABI of the B200-native reconstruction hot path
 * (disparity filter -> Q reprojection -> rigid transform -> VoxelGrid downsample -> global-cloud merge).
 *
 * This is the drop-in boundary for pk17r/online_3d_reconstruction.  The reference has no FFI of its
 * own; the seam is the set of `Pose` member calls listed below (file:line are relative to the
 * reference root).  Every entry point takes plain pointers and sizes, returns an int status
 * (0 = ok, <0 = error, message via o3r_last_error) and never throws across the boundary; the
 * reference's per-frame catch-all (pose.cpp:620-635) maps any failure to "empty cloud + message",
 * which is what a caller gets by treating a negative status as n_out = 0.
 *
 * There is NO CPU fallback behind this interface: every compute entry point runs hand-written
 * sm_100a CUDA kernels and fails with O3R_ERR_CUDA when no usable device is present.
 */
#ifndef O3R_H
#define O3R_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define O3R_VERSION 1

/* ---- status codes ------------------------------------------------------------------------- */
#define O3R_OK               0
#define O3R_ERR_INVALID     -1   /* bad argument / parameter combination                        */
#define O3R_ERR_CUDA        -2   /* CUDA runtime error or no device                             */
#define O3R_ERR_CAPACITY    -3   /* caller's output buffer too small (n_out still reports need) */
#define O3R_ERR_UNSUPPORTED -4   /* operation not available in the context's merge mode         */
#define O3R_ERR_NOMEM       -5

/* ---- record types -------------------------------------------------------------------------- */

/* pcl::PointXYZRGB as it crosses the boundary (SURVEY §8a row P): the reference's 32-byte PCL
 * record carries 16 bytes of information; colour is 0x00RRGGBB packed exactly as
 * pose_functions.cpp:1083/1120 does from the BGR Vec3b (alpha byte 0). */
typedef struct o3r_point {
    float    x, y, z;
    uint32_t rgb;
} o3r_point;

/* Cell record: partial sums on the combined grid.  Exchanged between ranks (o3r_exchange_cycle) and, bit for bit the
 * resident accumulators, the record of a map checkpoint (o3r_cloud_export_cells / o3r_cloud_import_cells). */
typedef struct o3r_cell {
    uint64_t key;            /* (k+2^20)<<42 | (j+2^20)<<21 | (i+2^20) */
    float    sx, sy, sz;     /* sums of x, y, z+500 (float)            */
    uint32_t n;              /* points in the partial                   */
    uint32_t sr, sg, sb;     /* colour sums                             */
    uint32_t pad;
} o3r_cell;                  /* 40 bytes */

/* disparity sample formats.  U8 is the reference's native format (pose_functions.cpp:548,1104);
 * F64 is the plane-fitted image of --use_segment_labels (pose_functions.cpp:905,1102);
 * U16 (value / disp_divisor, the commented variant at pose_functions.cpp:1102) and F32 are the
 * north-star extensions. */
enum { O3R_DISP_U8 = 0, O3R_DISP_U16 = 1, O3R_DISP_F32 = 2, O3R_DISP_F64 = 3 };

/* blur applied when blur_kernel > 1 (pose_functions.cpp:1040-1047).  The reference's live filter is
 * cv::bilateralFilter(src, dst, k, 2k, k/2) (pose_functions.cpp:1044, integer k/2); north_star names median
 * (the commented alternative at :1045) and box. */
enum { O3R_BLUR_MEDIAN = 0, O3R_BLUR_BOX = 1, O3R_BLUR_BILATERAL = 2 };

/* how the global cloud is kept (SURVEY §8a row M) */
enum {
    O3R_MERGE_ACCUMULATE = 0, /* per-cell accumulators keyed by the combined-grid key, merged every
                                 cycle; o3r_cloud_transform is unsupported.  Colour sums are exact
                                 uint32 (PCL folds floats: the colours differ once a cell's channel
                                 sum passes 2^24, ~65 800 points).  PCL's int32 guard is NOT emulated on
                                 the combined grid: a map wider than 2^31 combined cells still gets
                                 cells where the reference would return cloud_big unchanged.  Cells are
                                 limited to +-(2^20 - 1) per axis                                   */
    O3R_MERGE_RETAIN     = 1, /* cloud_big kept as points (pose.cpp:434); o3r_cloud_transform
                                 applies tf_icp in place (pose.cpp:353); one-shot voxelisation     */
    O3R_MERGE_ACCUMULATE_TILED = 2, /* as ACCUMULATE, but every 1024 consecutive per-frame voxels are first
                                 summed per cell inside the GPU's shared memory and only those partial
                                 sums are sorted and merged (8x less traffic).  Cell keys, point counts and
                                 colour sums are identical to ACCUMULATE; centroids differ by float
                                 reassociation only (<= 1e-5 relative, north_star's tolerance) and are
                                 reproducible from run to run.  While the pre-reduction does not reduce
                                 (more than one partial per two voxels: grids finer than the point spacing)
                                 it is skipped and the voxels are merged directly, as in ACCUMULATE    */
    O3R_MERGE_ACCUMULATE_FUSED = 3 /* the fused disparity -> cloud -> voxel pipeline: the per-frame clouds are never written to
                                 memory.  Three engines serve it, best first (o3r_last_batch_engine):
                                 2 tile   — dense scans (jump_pixels 1, no keypoints) of a rectified-stereo Q: ONE kernel from
                                            the disparity / colour planes to per-cell partial sums; a tile of 64 x 32 pixels and
                                            its halo are evaluated into shared memory, the points of a per-frame leaf are found
                                            in a small pixel window around the leaf's first point and summed in scan order
                                            (per-frame VoxelGrid centroids bit-identical to ACCUMULATE's), and the centroids
                                            are summed per combined cell inside the tile;
                                 1 bucket — strided scans, keypoints, rows that are not 4-aligned, leaves wider than the
                                            widest pixel window: points are binned once into buckets of 5 x 5 leaf columns
                                            and every bucket is finished in shared memory;
                                 0 sort   — everything else (StatisticalOutlierRemoval on, a Q without the rectified-stereo
                                            sparsity, device-side limits of the other two exceeded, a combined grid so fine
                                            that nothing reduces): runs as ACCUMULATE_TILED.
                                 o3r_last_batch_points is unsupported while engines 1 / 2 serve the batch (frame_counts are
                                 still reported).  Same result contract as ACCUMULATE_TILED: keys, counts, colour sums exact,
                                 centroids within float reassociation (<= 1e-5 relative), reproducible bit for bit           */
};

/* Read-only configuration: the `Pose` members the path reads (pose.h:93-98,108,118,126-128,149,168). */
typedef struct o3r_params {
    int      rows, cols;              /* pose.h:95 (set from the first image, pose_functions.cpp:636) */
    int      cols_start_aft_cutout;   /* pose.h:95 = cols / cutout_ratio (pose_functions.cpp:638)     */
    int      bounding_box;            /* pose.h:94 (20)                                               */
    double   min_disparity;           /* pose.h:93 (64): valid iff (double)disp > min_disparity       */
    double   Q[16];                   /* pose.h:128, row-major 4x4 double                             */
    int      jump_pixels;             /* pose.h:96: 0 = keypoints only, 1 = dense grid, J = stride    */
    int      blur_kernel;             /* pose.h:98: <= 1 = off                                         */
    int      blur_mode;               /* O3R_BLUR_*                                                    */
    double   voxel_size;              /* pose.h:118                                                    */
    unsigned min_points_per_voxel;    /* pose.h:108 (combined grid only, pose_functions.cpp:1693)     */
    int      dont_downsample;         /* pose.h:149                                                    */
    int      use_segment_labels;      /* pose.h:168: disparity is F64, or labels + plane coefficients */
    double   disp_divisor;            /* U16 only: disp = (double)raw / disp_divisor (200.0)          */
    int      merge_mode;              /* O3R_MERGE_*                                                   */
    int      device;                  /* CUDA device ordinal                                           */
    int      max_batch_frames;        /* frames the context sizes its staging buffers for (>=1)       */
    int      sor_mean_k;              /* pcl::StatisticalOutlierRemoval before the per-frame VoxelGrid
                                         (pose_functions.cpp:1673-1686; the reference uses 50 whenever
                                         jump_pixels > 0).  0 = filter off                             */
    double   sor_stddev_mul;          /* setStddevMulThresh (1.0 in the reference)                     */
} o3r_params;

/* One frame of input: what createAndTransformPtCloud reads from acceptedImageDataVec[i]
 * (pose.cpp:596-607, pose_functions.cpp:1035-1051).  Pointers are host or device memory according
 * to the entry point used. */
typedef struct o3r_frame {
    const void*    disp;          /* rows x cols samples of disp_type, row stride disp_step BYTES  */
    size_t         disp_step;
    const uint8_t* bgr;           /* rows x cols x 3 (cv::Mat CV_8UC3, BGR), row stride bgr_step    */
    size_t         bgr_step;
    const uint8_t* labels;        /* optional rows x cols u8 segment labels (with plane_coef)       */
    size_t         labels_step;
    const double*  plane_coef;    /* optional [n_planes][3] = (a,b,c): disp = a*x + b*y + c for
                                     label l = index+1; label 0 / label > n_planes -> 0.0
                                     (pose_functions.cpp:968-971)                                   */
    int            n_planes;
    const float*   kp_xy;         /* optional ORB keypoints, n_kp pairs (x,y) (pose_functions.cpp:1059) */
    int            n_kp;
    float          T[16];         /* t_mat_FeatureMatched, row-major float 4x4 (pose.h:83)          */
} o3r_frame;

typedef struct o3r_ctx o3r_ctx;

/* ---- lifecycle ------------------------------------------------------------------------------ */

/* Replaces: construction of the read-only Pose state after populateData (pose.cpp:23-127). */
int  o3r_create(const o3r_params* params, o3r_ctx** out_ctx);
void o3r_destroy(o3r_ctx* ctx);
const char* o3r_last_error(const o3r_ctx* ctx);   /* ctx may be NULL: last create() error */
int  o3r_version(void);

/* Page-locked host memory for image buffers handed to the host-pointer entry points: copies from it run
 * at full PCIe rate and asynchronously (what cv::cuda::HostMem would give the reference's cv::Mat). */
void* o3r_host_alloc(size_t bytes);
void  o3r_host_free(void* p);

/* ---- per-frame path --------------------------------------------------------------------------- */

/* Replaces: void Pose::createAndTransformPtCloud(int, PointCloud::Ptr&)  pose.cpp:596-636
 *   = createSingleImgPtCloud (pose_functions.cpp:1030-1134) + transformPtCloud (:1358-1362)
 *   + downsamplePtCloud(cloud,false) (:1654-1709: StatisticalOutlierRemoval when sor_mean_k > 0, then VoxelGrid leaf
 *     voxel_size/5).
 * Host pointers in `frame`; `out` is a host buffer of `cap` records; *n_out = records produced
 * (also set on O3R_ERR_CAPACITY).  Output order is the reference's: keypoints then row-major grid
 * (dont_downsample) or ascending VoxelGrid index.  Thread-safe per ctx (internally serialised). */
int o3r_frame_cloud(o3r_ctx* ctx, const o3r_frame* frame, int disp_type,
                    o3r_point* out, size_t cap, size_t* n_out);

/* Replaces: the cycle's fan-out + ordered concat + append, pose.cpp:361-434:
 *   for each accepted frame createAndTransformPtCloud, concatenate in frame order, cloud_big.insert.
 * Runs the n frames as one batched launch sequence and appends/merges the result into the
 * resident cloud.  Host pointers; only the scan ROI of each plane is copied, on the context's copy streams, overlapping
 * compute.  Consecutive frames whose disparity AND colour planes sit back to back in host memory with one row pitch
 * (frames[i+1].disp == frames[i].disp + rows * disp_step, same for bgr: a cycle kept in one o3r_host_alloc arena, the
 * equivalent of the reference's rawImageDataVec in page-locked memory) are moved with one 3-D copy per plane type and group
 * of up to 16 frames (extent = the ROIs of the group's planes) — ~13 % less copy time than one 2-D copy per plane.
 * If frame_counts != NULL it receives each frame's output record count (n entries). */
int o3r_frames_cloud(o3r_ctx* ctx, const o3r_frame* frames, int n, int disp_type,
                     uint32_t* frame_counts);

/* Announces the frames of a coming o3r_frames_cloud call (same frame pointers, same n) so that their host->device copies
 * overlap whatever the context is computing (input staging is double-buffered: one prefetch may be pending while the call
 * before it is issued, e.g. prefetch(k+1); frames_cloud(k); ...).  The request is only recorded here; the copies are issued
 * on the context's copy streams by the next frame-path call (right after its kernels are queued) or the next prefetch.
 * The reference loads every image into host RAM up front (populateData, pose_functions.cpp:624-744); this is the
 * device-side equivalent for the next cycle.
 * LIFETIME: from this call on the library may read the frames' host buffers at any time, until either the matching
 * o3r_frames_cloud call (same buffer pointers, n and disp_type) has returned or o3r_frames_prefetch_cancel has returned;
 * they must stay allocated and unchanged for that long.  A prefetch is matched by its buffer POINTERS, so buffers that are
 * recycled with new contents before then would be served stale.  A prefetch that is never consumed only costs the copy —
 * but its buffers stay bound by the rule above until it is cancelled or overwritten by two later prefetches. */
int o3r_frames_prefetch(o3r_ctx* ctx, const o3r_frame* frames, int n, int disp_type);

/* Abandons every announced prefetch: a recorded request is dropped, copies already in flight are waited for, staged inputs
 * are forgotten.  When it returns the library holds no reference to any prefetched host buffer. */
int o3r_frames_prefetch_cancel(o3r_ctx* ctx);

/* Same as o3r_frames_cloud but every pointer inside `frames` is DEVICE memory on ctx's device and
 * nothing is copied (the inputs-resident-in-HBM measurement).  T is still read from host. */
int o3r_frames_cloud_dev(o3r_ctx* ctx, const o3r_frame* frames, int n, int disp_type,
                         uint32_t* frame_counts);

/* Copies the last batch's concatenated per-frame clouds (what was appended) to the host. */
int o3r_last_batch_points(o3r_ctx* ctx, o3r_point* out, size_t cap, size_t* n_out);

/* ---- global cloud ----------------------------------------------------------------------------- */

/* Replaces: transformPtCloud(cloud_big, cloud_big, tf_icp)  pose.cpp:350-354 (RETAIN mode only). */
int o3r_cloud_transform(o3r_ctx* ctx, const float T[16]);

/* Replaces: cloud_big->insert(end, ...) pose.cpp:434 for points produced elsewhere
 * (e.g. the --downsample tool reading a PLY, pose.cpp:71-77).  Host pointer.  In the accumulate modes a point
 * outside +-(2^20 - 1) combined-grid cells on any axis, or with a NaN / inf coordinate, makes the call return
 * O3R_ERR_INVALID without merging any of the n points. */
int o3r_cloud_append(o3r_ctx* ctx, const o3r_point* pts, size_t n);

/* Replaces: PointCloud::Ptr Pose::downsamplePtCloud(PointCloud::Ptr&, bool combinedPtCloud=true)
 *   pose_functions.cpp:1654-1709, callers pose.cpp:530 (final), :645 (preview), :77 (--downsample).
 * z += 500, VoxelGrid leaf (v, v, 1000), min_points_per_voxel, z -= 500; output ascending voxel
 * index.  With dont_downsample the cloud itself is returned (pose.cpp:535).  The resident cloud is
 * left untouched.  `out` may be NULL with cap = 0 to query the size. */
int o3r_cloud_downsample(o3r_ctx* ctx, o3r_point* out, size_t cap, size_t* n_out);

/* Same, but the result stays on the GPU: *dev_out points at *n_out records in device memory owned by the
 * context (valid until the next call on it) — for consumers on the same device (a CUDA viewer, the next
 * pipeline stage) and for the inputs-resident-in-HBM measurement. */
int o3r_cloud_downsample_dev(o3r_ctx* ctx, const o3r_point** dev_out, size_t* n_out);

/* Number of resident records (cells in ACCUMULATE mode, points in RETAIN mode) and clear. */
int o3r_cloud_size(o3r_ctx* ctx, size_t* n);
int o3r_cloud_clear(o3r_ctx* ctx);

/* Change tracking of the resident cloud (O3R_MERGE_ACCUMULATE, _TILED, _FUSED; with or without a communicator): a
 * consumer that keeps a copy of the combined grid (a viewer, a link to a ground station, the next pipeline stage) reads
 * after each cycle only the cells that cycle touched instead of the whole map.  Upserting the records by key into a
 * key-sorted map keeps that map equal to o3r_cloud_downsample's output, order included.
 *   - Tracking.  enable = 1 starts tracking, or restarts it when it is on; the next o3r_cloud_changes then returns every
 *     cell the downsample would emit (the full state: how a consumer that joins late or reconnects starts).  enable = 0
 *     stops tracking and frees its buffers.  Tracking is off by default; while it is off it costs nothing.  While it is
 *     on, every merged cycle adds four small kernel launches and nothing is read back.
 *   - Records.  A call returns every cell whose point count grew since the last consuming call and whose count is
 *     >= min_points_per_voxel, and no other cell (except the full state after an enable), in ascending cell key (=
 *     ascending voxel index).  Each record is bit-identical to that cell's record in o3r_cloud_downsample.  keys (the
 *     absolute cell key, as o3r_voxel_grid reports it) and counts (points in the cell) are optional; either may be NULL.
 *   - Query, then fill.  out = NULL with cap = 0 queries *n_out and consumes nothing (a second query returns the same
 *     records).  A call that delivers the records and returns O3R_OK consumes them; O3R_ERR_CAPACITY consumes nothing and
 *     still reports *n_out.  A merge, clear or enable between the query and the fill makes the fill return the grown set.
 *     The query's result is kept until the tracked state changes, so query-then-fill computes it once.
 *   - o3r_cloud_changes_dev: the records stay in device buffers owned by the context, valid until the next call on it;
 *     the call consumes on return.  Any of the three pointers may be NULL.
 *   - o3r_cloud_clear empties the pending set; tracking stays as it was (a consumer that clears the cloud clears its map).
 *   - With a communicator each rank returns the changes of the cells it owns; the union over ranks is the global change
 *     set.  After an exchange slot overflow o3r_cloud_changes fails with O3R_ERR_CAPACITY (the next o3r_cloud_downsample
 *     still reports the overflow too).
 *   - O3R_MERGE_RETAIN and dont_downsample: O3R_ERR_UNSUPPORTED from all three calls (every transform moves every point,
 *     so there is no cheap change set).  o3r_cloud_changes[_dev] with tracking off: O3R_ERR_INVALID. */
int o3r_cloud_track_changes(o3r_ctx* ctx, int enable);
int o3r_cloud_changes(o3r_ctx* ctx, o3r_point* out, uint64_t* keys, uint32_t* counts, size_t cap, size_t* n_out);
int o3r_cloud_changes_dev(o3r_ctx* ctx, const o3r_point** dev_out, const uint64_t** dev_keys,
                          const uint32_t** dev_counts, size_t* n_out);

/* Checkpoints of the resident map: a map outlives its context (a survey resumed after a restart, two flights merged, a
 * shard moved to another number of GPUs).  The library does no file I/O; host/mapfile.hpp and mapfile.py define a file.
 *   - o3r_cloud_export_cells (O3R_MERGE_ACCUMULATE, _TILED, _FUSED without dont_downsample): every resident cell in ascending
 *     key, cells below min_points_per_voxel included (they are state: a later cycle can lift them over the threshold).  Each
 *     field is a bit copy of the accumulators; pad is 0.  Query, then fill, as o3r_cloud_downsample: out = NULL with cap = 0
 *     reports *n_out; a short buffer returns O3R_ERR_CAPACITY with *n_out set.  With a communicator each rank exports the
 *     shard it owns; a batch still waiting for its o3r_exchange_cycle is not in that shard yet.
 *   - o3r_cloud_import_cells (same modes): merges the n records as ONE cycle through the ordinary merge.  A resident cell,
 *     and a key that appears more than once, gets the imported sums added in input order after the resident sums; importing
 *     an export into an empty context reproduces it bit for bit, and a resumed run ends where the uninterrupted one does: bit
 *     for bit in O3R_MERGE_ACCUMULATE; in _TILED / _FUSED bit for bit when the batches are merged the same way, but these
 *     modes pick the engine (and whether to pre-reduce) from the context's own batch history, which a checkpoint does not
 *     carry, so a resumed map may differ in the centroids within the mode's float-reassociation contract.  Host pointer, copied before the call returns.  The
 *     records are staged in a buffer of their own: the last batch (o3r_last_batch_points, a pending o3r_exchange_cycle) is
 *     left intact.  All or nothing: every record is checked on the device first, and if any is refused the call returns
 *     O3R_ERR_INVALID, merges nothing, and o3r_last_error names the first refused index and its reasons.  A record is
 *     refused when bit 63 of its key is set, a 21-bit key field is 0 (outside +-(2^20 - 1) cells), n == 0, sx / sy / sz is
 *     not finite, a colour sum exceeds 255 * n, pad != 0, or (with a communicator) hash64(key) % world != rank.  Whether a
 *     centroid lies inside its key's cell is not checked: rounding of a genuine sum / n can land it across the boundary.
 *     With change tracking on, the cells the import grew become pending changes like those of any merge.
 *   - o3r_cloud_export_points (O3R_MERGE_RETAIN, or any mode with dont_downsample): cloud_big in order, exactly; query then
 *     fill as above.  o3r_cloud_append is the matching import.
 *   - O3R_ERR_UNSUPPORTED: the cell calls outside their modes, o3r_cloud_export_points outside its modes or with a
 *     communicator attached (a sharded point cloud carries frame-order tags a checkpoint cannot carry). */
int o3r_cloud_export_cells(o3r_ctx* ctx, o3r_cell* out, size_t cap, size_t* n_out);
int o3r_cloud_import_cells(o3r_ctx* ctx, const o3r_cell* cells, size_t n);
int o3r_cloud_export_points(o3r_ctx* ctx, o3r_point* out, size_t cap, size_t* n_out);

/* ---- stand-alone stages (parity probes; same kernels as above) ------------------------------- */

/* pcl::VoxelGrid<PointXYZRGB>::filter on a host cloud: leaf (lx,ly,lz) as PCL's setLeafSize floats,
 * min_points as setMinimumPointsNumberPerVoxel.  Optional outputs: keys[n_out] = the 64-bit absolute
 * cell key (SURVEY §8a row VG), counts[n_out] = points per emitted voxel, *passthrough = 1 when PCL's
 * int32 overflow guard returned the input unchanged. */
int o3r_voxel_grid(o3r_ctx* ctx, const o3r_point* pts, size_t n, float lx, float ly, float lz,
                   unsigned min_points, o3r_point* out, size_t cap, size_t* n_out,
                   uint64_t* keys, uint32_t* counts, int* passthrough);

/* pcl::StatisticalOutlierRemoval alone on a host cloud (pose_functions.cpp:1673-1686: setMeanK(50),
 * setStddevMulThresh(1.0)): keep[i] = 0 for the points PCL removes; dist (optional, n floats) = every point's mean
 * distance to its mean_k nearest neighbours; threshold (optional) = mean + mul * stddev of those. */
int o3r_sor(o3r_ctx* ctx, const o3r_point* pts, size_t n, int mean_k, double stddev_mul,
            uint8_t* keep, float* dist, double* threshold);

/* The blur stage alone on a u8 plane (pose_functions.cpp:1040-1047 with blur_mode). Host pointers. */
int o3r_blur_u8(o3r_ctx* ctx, const uint8_t* src, size_t src_step, int rows, int cols,
                int kernel, int mode, uint8_t* dst, size_t dst_step);

/* ---- pre-pass: the per-frame reductions in front of the hot path (SURVEY 8f-3) --------------------------- */

/* Replaces: double Pose::getVariance(Mat disp_img, false) (pose_functions.cpp:1007-1028, with getMean :987-1005):
 * the bad-frame gate of the accept loop (pose.cpp:187-196 rejects a frame whose variance is > 5).  The reference's
 * formula is kept as written: sums run over the VALID ROI samples (disp > min_disparity) but are divided by ALL ROI
 * samples (minus one for the variance).  u8 disparity, host pointer. */
int o3r_disp_variance(o3r_ctx* ctx, const uint8_t* disp, size_t disp_step, double* variance);

/* Replaces: void Pose::createPlaneFittedDisparityImages(int) (pose_functions.cpp:900-985): for every segment label
 * 1, 2, ... (until the first label that does not occur, :923) the least-squares plane d = a*x + b*y + c over the
 * label's pixels strictly inside the ROI (:929), solved as inv_SVD(AtA) * At * b (:957-965).  coef receives
 * [n_planes][3] doubles (coef_cap = planes it can hold, 255 suffices for 8-bit labels); a label without ROI pixels
 * keeps (0, 0, 0) (:939-940).  The result is what o3r_frame.plane_coef takes.  If variance != NULL it receives
 * getVariance(plane-fitted image, true) (:973); the reference throws when it exceeds 3 (:975-982). */
int o3r_plane_fit(o3r_ctx* ctx, const uint8_t* labels, size_t labels_step, const uint8_t* disp, size_t disp_step,
                  double* coef, int coef_cap, int* n_planes, double* variance);

/* Per-pixel validity mask of the grid scan (1 byte per scanned pixel, row-major over the ROI
 * samples) for one frame — the bit-exact mask contract of north_star. Host pointers. */
int o3r_frame_mask(o3r_ctx* ctx, const o3r_frame* frame, int disp_type,
                   uint8_t* mask, size_t cap, size_t* n_scanned);

/* ---- multi-GPU exchange (SURVEY §8e) ---------------------------------------------------------- */

/* Parity probe for O3R_MERGE_ACCUMULATE_FUSED: when set, the fused engine also stores every per-frame voxel centroid of
 * the batch, in no particular order, and o3r_last_batch_points returns that multiset. */
int o3r_set_keep_frame_voxels(o3r_ctx* ctx, int keep);

/* ---- the exchange inside the library -------------------------------------------------------------------------------------
 * One process per GPU; rank r reconstructs the cycle's frames f with f mod world == r (the reference's 7-thread fan-out,
 * pose.cpp:383-424, spread over GPUs) and owns the combined-grid cells whose hash64(key) mod world == r.  After each
 * o3r_frames_cloud* call every rank calls o3r_exchange_cycle: the batch is pre-reduced on the combined grid (one record per
 * distinct cell of the cycle), the cells are bucketed by owner and exchanged with grouped ncclSend / ncclRecv on the context's
 * stream, and what arrives is folded into the rank's shard.  Each (source, destination) pair moves ONE fixed-size slot of
 * slot_cells cells per cycle with the valid count in its first record, so nothing about a cycle's exchange crosses the host
 * and the call returns without waiting for the GPU.  slot_cells must be the same on all ranks; size it at twice the cells one
 * rank sends to one owner in a cycle (the distinct combined-grid cells of a rank's cycle / world — o3r_cloud_size after one
 * probe cycle).  An overflowing slot drops cells: the next o3r_cloud_downsample then fails with O3R_ERR_CAPACITY.
 * The union of the ranks' o3r_cloud_downsample outputs, ordered by cell key, is the single-GPU cloud: keys, counts and
 * colours exactly, centroids within float reassociation (1e-5 relative).
 * NCCL is loaded at run time (libnccl.so.2); o3r_comm_unique_id + o3r_comm_init create a communicator of the library's own
 * (the id travels by whatever channel the host has: MPI, a file, torch.distributed), o3r_comm_attach adopts an existing
 * ncclComm_t.  While a communicator is attached, o3r_frames_cloud* leaves the merge to o3r_exchange_cycle; after
 * o3r_comm_destroy the context merges its cycles itself again.
 *
 * O3R_MERGE_RETAIN (ICP on) and dont_downsample shard differently: the points stay on the rank that made them.
 *   - o3r_comm_init / o3r_comm_attach need an empty resident cloud (O3R_ERR_INVALID otherwise); slot_cells is checked but
 *     not used, no slot buffers are allocated.
 *   - Every o3r_frames_cloud* call appends the rank's frames (f mod world == rank, in order) to its local cloud and counts
 *     as one cycle, so all ranks make the same number of calls; n = 0 is a cycle in which this rank has no frame.
 *   - o3r_cloud_transform stays local: every rank applies the same T at the same point of the call sequence.
 *   - o3r_exchange_cycle is a no-op returning O3R_OK; o3r_cloud_append returns O3R_ERR_UNSUPPORTED (appended points have
 *     no place in the global frame order); o3r_cloud_size and o3r_cloud_clear stay local (all ranks clear together).
 *   - o3r_cloud_downsample / o3r_cloud_downsample_dev are collectives: the global bbox is all-reduced, every point travels
 *     once to the owner of its combined-grid cell (hash64(absolute cell key) mod world) with an order tag (cycle, global
 *     frame), and the owner sums its cells' points in cloud_big order.  Each rank returns the cells it owns, ascending
 *     voxel index, min_points_per_voxel applied; the union ordered by key is the single-GPU output bit for bit, centroids
 *     included.  On a pass-through grid (PCL's int32 guard on the GLOBAL bbox) and with dont_downsample every rank returns
 *     its own points, which, interleaved back in frame order, are the single-GPU output.  The result is kept until the local
 *     cloud changes (frames, transform, clear): a second call (the cap = 0 query, then the fill) does not communicate.
 *     A rank that fails takes part in every agreement step, so all ranks return an error and none is left waiting.
 *     Limits: fewer than 2^32 points per rank and per owner; bits(cycles) + bits(frames per cycle) <= 32 (the order tag),
 *     beyond which every rank returns O3R_ERR_UNSUPPORTED; clear the cloud to start the count again. */
#define O3R_COMM_ID_BYTES 128
int o3r_comm_unique_id(void* id_out /* O3R_COMM_ID_BYTES, rank 0 */);
int o3r_comm_init(o3r_ctx* ctx, int world, int rank, const void* id, size_t slot_cells);   /* collective */
int o3r_comm_attach(o3r_ctx* ctx, void* nccl_comm, int world, int rank, size_t slot_cells);
int o3r_comm_destroy(o3r_ctx* ctx);
int o3r_exchange_cycle(o3r_ctx* ctx);                                                     /* collective, asynchronous */

/* ---- introspection ----------------------------------------------------------------------------- */

/* Per-kernel CUDA-event timing on the context's stream.  o3r_profile(ctx, 1) starts recording an event
 * pair around every kernel launch; o3r_profile_read writes one line per kernel name,
 * "name<TAB>launches<TAB>total_ms", into buf.  o3r_profile(ctx, 0) stops and clears. */
int o3r_profile(o3r_ctx* ctx, int enable);
int o3r_profile_read(o3r_ctx* ctx, char* buf, size_t cap);

/* Kernel launches issued by this context so far (bench.py's gpu_launches). */
uint64_t o3r_launch_count(const o3r_ctx* ctx);
/* Partial cells the last batch produced (O3R_MERGE_ACCUMULATE_TILED / _FUSED; 0 otherwise): the record count the
 * merge's sort and reduce ran on, for traffic accounting. */
size_t o3r_last_batch_partials(const o3r_ctx* ctx);
/* Engine the last batch ran through: 2 = the tile engine, 1 = the bucket engine (both O3R_MERGE_ACCUMULATE_FUSED only),
 * 0 = the sort engine (every other mode, and FUSED batches the other two could not take). */
int o3r_last_batch_engine(const o3r_ctx* ctx);
/* The CUDA stream all work of the context is issued on (a cudaStream_t) — for event timing. */
void* o3r_stream(o3r_ctx* ctx);
/* Blocks until all work issued on the context's stream has completed. */
int o3r_sync(o3r_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* O3R_H */
