// tile.cuh — the fused tile engine of O3R_MERGE_ACCUMULATE_FUSED: ONE kernel from the disparity / colour planes to the
// partial sums of the combined grid.
//
// What it replaces: createSingleImgPtCloud (pose_functions.cpp:1030-1134) + transformPtCloud (:1358-1362) +
// downsamplePtCloud(cloud, false) (:1654-1709, pcl::VoxelGrid with leaf voxel_size / 5) + the append to cloud_big
// (pose.cpp:434) of a whole cycle, up to the per-cell partial sums that the incremental merge (voxel.cuh engine 2) folds
// into the resident shard — the dense scan (jump_pixels == 1, no keypoints) of a rectified-stereo Q.
//
// Why no sort and no binning pass: inside ONE frame all points come from one projection centre, so the points of a leaf
// (a cube of edge voxel_size / 5) lie on rays that pass through that cube: they are pixels within a few columns and rows of
// each other.  Two points of one leaf differ by less than the leaf edge e on every world axis; in the camera frame
// dC = M^-1 dP (M = the frame's matrix), so |dX| <= e s_x, |dZ| <= e s_z with s = the absolute row sums of M^-1.  With the
// homogeneous coordinate w = q14 d + q15 (depth Z = q11 / w) and t2 = X2 / Z2:
//     |x1 - x2| = |q11 / q0| |X1/Z1 - X2/Z2| = |q11 / q0| |dX - t2 dZ| / |Z1| <= e (s_x + |t2| s_z) |w1| / |q0|,
// and the same in y.  With L = the worst e (s + t s_z) / |q| over the batch's matrices and the scan region, every leaf-mate
// of a pixel with |w| < (R + 1) / L lies in its (2R+1) x (2R+1) pixel window.  The host picks R from that bound, and the kernel
// checks it for every valid pixel it evaluates: a violation raises TV_FLAG_RANGE and the host reruns the batch with a larger
// window, or through the bucket engine (bucket.cuh).
//
// One CTA per tile of 64 x 32 pixels (ticket order = frame, tile row, tile column):
//   A  evaluate the tile plus a halo of R rows / 4 columns (validity, Q reprojection, rigid transform, colour, leaf cell):
//      planes {cell hash, x, y, z, rgb} in shared memory; the exact PCL bbox of the frame (atomicMin / Max) on the side
//   B  every core pixel compares the hashes of its window: an equal hash EARLIER in scan order (verified on the cell itself)
//      means the pixel is not its leaf's first point; a first point left-folds its later window mates in scan order — the
//      oracle's stable order, so the per-frame VoxelGrid centroid is bit-identical — and divides (pcl::CentroidPoint).
//      A leaf belongs to the tile that holds its first point, and the halo shows that tile every mate.
//   C  the centroids are celled on the combined grid (voxel_size, voxel_size, 1000 after z += 500); the tile's cells index
//      a dense table (no hash), the centroids are counting-sorted by cell (warp match + warp-private counters: no atomics)
//      and every cell is summed by four lanes in a fixed tree: one 40-byte partial cell per (tile, cell), in cell order.
//      (A tile whose cells span more than the table — a depth discontinuity, a grid finer than the pixels — writes every
//      centroid as its own single-point record instead.)
//   The records of a tile go to a scratch list at a position taken from an atomic cursor — no tile ever waits for another —
//   and k_tv_compact then copies them into the partial list in TILE order (a scan over the per-tile counts), so the list the
//   merge sees, and with it every float sum, is reproducible bit for bit.  (A decoupled look-back inside the kernel was
//   measured first: 14 % of the issued instructions were the spin on slower predecessors, plus the CTA-wide wait behind it.)
//
// PCL's int32 overflow guard (output = input for a frame whose leaf grid has more than 2^31 cells) depends on the frame's
// exact bbox, which only exists once every pixel has been evaluated: the kernel runs on the host's per-frame guess, computes
// the bbox anyway, and k_tv_check compares the guard's verdict with the guess (TV_FLAG_PASS + the actual flags -> rerun).
//
// Contract = O3R_MERGE_ACCUMULATE_TILED's: per-frame centroids bit-exact, cells / counts / colour sums exact, combined
// centroids equal to the oracle's single left fold within float reassociation (<= 1e-5 relative).
#pragma once
#include "bucket.cuh"
#include "common.cuh"
#include "sort.cuh"
#include "stage_a.cuh"

namespace o3r {

#ifndef O3R_TV_H
#define O3R_TV_H 32
#endif
#ifndef O3R_TV_BINS
#define O3R_TV_BINS 512
#endif
#ifndef O3R_TV_THREADS
#define O3R_TV_THREADS 256
#endif
constexpr int kTvThreads = O3R_TV_THREADS;             // threads of a tile's CTA: the kernel is latency-bound, T ~ 0.27 + 2.24 / (resident
constexpr int kTvWarps = kTvThreads / 32;              // CTAs of 8 warps) ms on configs[1] — more warps per SM is what buys time
constexpr int kTvW = 64, kTvH = O3R_TV_H;              // core pixels of a tile
constexpr int kTvGroupsRow = kTvW / 4;                 // 4-pixel groups per core row
constexpr int kTvCoreGroups = kTvGroupsRow * kTvH;     // 512: two per thread
constexpr int kTvQ = kTvCoreGroups / kTvThreads;         // core groups per thread
constexpr int kTvItems = kTvW * kTvH;                  // centroids a tile can emit
constexpr int kTvBinsN = O3R_TV_BINS;                       // distinct combined-grid cells a tile can sum (more: one record per centroid)
template <int R>
struct TvBins { static constexpr int value = kTvBinsN; };
constexpr int kTvHash = 2 * kTvItems;                  // hash slots of the sparse cell table (load <= 0.5)
static_assert((kTvHash & (kTvHash - 1)) == 0 && kTvHash <= 65536, "hash slots: a power of two that a 16-bit cell number covers");
constexpr int tv_log2(int v) { return v <= 1 ? 0 : 1 + tv_log2(v >> 1); }
constexpr int kTvHashShift = 32 - tv_log2(kTvHash);
constexpr int kTvMaxR = 4;
constexpr uint32_t kTvNoHash = 0xffffu;                // invalid pixel (valid hashes keep 15 bits; the plane holds 16-bit words)
static_assert(kTvQ * kTvThreads == kTvCoreGroups, "core groups must divide evenly");

enum { TV_FLAG_RANGE = 1u, TV_FLAG_SPACE = 2u, TV_FLAG_PASS = 4u };

template <int R>
struct TvGeom {
    static constexpr int HX = R ? 4 : 0, HY = R;       // halo columns stay a multiple of 4: aligned 4-pixel groups
    static constexpr int NC = kTvW + 2 * HX, NR = kTvH + 2 * HY, N = NC * NR, NG = N / 4;
    static constexpr int W = 2 * R + 1, S = R * W + R; // window width, index of the pixel itself
    // the planes (R > 0), later the sparse cell table (8-byte keys + 2-byte cell numbers), later the centroids in cell order
    static constexpr size_t alias_bytes = (size_t)kTvHash * 10 > (size_t)kTvItems * 16 ? (size_t)kTvHash * 10 : (size_t)kTvItems * 16;
    static constexpr size_t plane_bytes = (R && (size_t)N * 18 > alias_bytes) ? (size_t)N * 18 : alias_bytes;   // 2-byte hash + x, y, z, rgb
};

// mask of a pixel's later window positions: R (2R + 2) bits
template <int R>
struct TvMask { typedef uint32_t type; };
template <>
struct TvMask<4> { typedef unsigned long long type; };

template <int NB, int MB>
struct TvTail {
    static_assert(NB % kTvThreads == 0, "cells per thread");
    union {
        uint16_t cnt[kTvWarps][NB + 2];        // phase C: per warp and cell: count, then exclusive prefix over the warps
        struct { double rl[256]; float zl[256]; } lut;   // phase A
        unsigned long long ml[kTvItems * MB / 8];   // phase B: per core pixel the mask of its verified later mates (MB bytes each)
    } u;
    uint32_t bd[NB + 1];                     // per cell: first item | rank among the non-empty cells << 16
    uint32_t scan[34];
    uint32_t ticket, out0, nb, nitems, nbh;
    uint16_t off[40];                        // plane offset of the window's later position k (TvLater::offset, tabulated: the
                                             // division by the window width cost ~8 instructions per verified / folded mate)
    int cmin[3], cmax[3];
    uint32_t bb[6];
    uint32_t any_valid, bad;
};
template <int R>
constexpr size_t tv_smem() { return TvGeom<R>::plane_bytes + sizeof(TvTail<TvBins<R>::value, (int)sizeof(typename TvMask<R>::type)>); }

// CTAs of this instantiation that fit an SM's 228 KB (1 KB reserved per CTA): the register budget follows from it
template <int R>
constexpr int tv_ctas_per_sm() {
    return (int)((size_t)233472 / (tv_smem<R>() + 1024)) < 1 ? 1 : (int)((size_t)233472 / (tv_smem<R>() + 1024)) > 4 ? 4
                                                                   : (int)((size_t)233472 / (tv_smem<R>() + 1024));
}

struct TvArgs {
    const FrameDev* frames;
    const uint8_t* frame_pass;     // the host's guess of PCL's overflow guard per frame
    int ntx, nty, n_frames;
    float inv_f, icx, icz;
    double wlim;                   // |q14 d + q15| must stay below this for the window to hold every leaf-mate
    int dlim_i;                    // the same bound as a u8 disparity (LUT path)
    o3r_cell* scratch;             // the chunk's records in arrival order
    uint32_t scratch_cap;
    uint32_t* cursor;              // next free scratch record
    uint32_t* tile_cnt;            // per tile (ticket order): records,
    uint32_t* tile_at;             // first scratch record
    uint32_t* ticket;
    uint32_t* frame_vox;
    uint32_t* bbox;
    int* cellbb;
    uint32_t* flags;
    float4* dbg_vox;
    uint32_t* dbg_cnt;
};

__device__ __forceinline__ uint32_t tv_hash(int i, int j, int k) {
    uint32_t h = (uint32_t)i * 0x9e3779b1u + (uint32_t)j * 0x85ebca77u + (uint32_t)k * 0xc2b2ae3du;
    h ^= h >> 15;
    return (h ^ (h >> 17)) & 0x7fffu;
}

// The thread's 4 consecutive pixels (xb .. xb + 3, y) of the dense scan: validity + camera-frame point, exactly the
// arithmetic of eval4's vector branch (stage_a.cuh).  `over` is raised when a valid pixel breaks the window bound.
template <int DT>
__device__ __forceinline__ uint32_t tv_eval4(const AParams& P, const FrameDev& F, const double* rl, const float* zl, int xb, int y,
                                             const TvArgs& A, float (&X)[4], float (&Y)[4], float (&Z)[4], bool& over) {
    uint32_t mask = 0;
    const uint8_t* row = F.disp + (size_t)y * F.disp_step;
    if (DT == O3R_DISP_U8) {
        const uint32_t w = *reinterpret_cast<const uint32_t*>(row + xb);
        if (P.use_lut) {
            const double vy = __dadd_rn(__dmul_rn(P.q[5], (double)y), P.q[7]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int d = (w >> (8 * j)) & 255;
                if (d > P.thr_i) {
                    mask |= 1u << j;
                    over = over || d > A.dlim_i;
                    const double s = rl[d];
                    const double v0 = __dadd_rn(__dmul_rn(P.q[0], (double)(xb + j)), P.q[3]);
                    X[j] = __double2float_rn(__dmul_rn(v0, s));
                    Y[j] = __double2float_rn(__dmul_rn(vy, s));
                    Z[j] = zl[d];
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int d = (w >> (8 * j)) & 255;
                if (d > P.thr_i) {
                    mask |= 1u << j;
                    double hw;
                    reproject_w(P, xb + j, y, (double)d, X[j], Y[j], Z[j], hw);
                    over = over || !(fabs(hw) < A.wlim);
                }
            }
        }
    } else {
        double dv[4];
        if (DT == O3R_DISP_U16) {
            const uint2 w = *reinterpret_cast<const uint2*>(row + 2 * (size_t)xb);
            dv[0] = __ddiv_rn((double)(w.x & 0xffffu), P.div); dv[1] = __ddiv_rn((double)(w.x >> 16), P.div);
            dv[2] = __ddiv_rn((double)(w.y & 0xffffu), P.div); dv[3] = __ddiv_rn((double)(w.y >> 16), P.div);
        } else if (DT == O3R_DISP_F32) {
            const float4 w = *reinterpret_cast<const float4*>(row + 4 * (size_t)xb);
            dv[0] = (double)w.x; dv[1] = (double)w.y; dv[2] = (double)w.z; dv[3] = (double)w.w;
        } else {
            const double2 a = *reinterpret_cast<const double2*>(row + 8 * (size_t)xb);
            const double2 b = *reinterpret_cast<const double2*>(row + 8 * (size_t)xb + 16);
            dv[0] = a.x; dv[1] = a.y; dv[2] = b.x; dv[3] = b.y;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (dv[j] > P.min_disp) {
                mask |= 1u << j;
                double hw;
                reproject_w(P, xb + j, y, dv[j], X[j], Y[j], Z[j], hw);
                over = over || !(fabs(hw) < A.wlim);
            }
    }
    return mask;
}

// The window positions LATER than a pixel in scan order, numbered in scan order: (0, 1..R), then rows 1..R with columns -R..R.
template <int R>
struct TvLater {
    static constexpr int W = 2 * R + 1, N = R + R * W;
    __device__ static __forceinline__ constexpr int bit(int dr, int dc) { return dr == 0 ? dc - 1 : R + (dr - 1) * W + (dc + R); }
    __device__ static __forceinline__ int offset(int k, int nc) {   // plane offset of position k
        if (k < R) return k + 1;
        const int q = k - R, dr = q / W;
        return (dr + 1) * nc + (q - dr * W) - R;
    }
};

// four consecutive masks as 16-byte shared-memory accesses (a lane's stride is 16 / 32 bytes: scalar accesses would conflict 4-way)
__device__ __forceinline__ void tv_st4(uint32_t* m, const uint32_t (&v)[4]) { *reinterpret_cast<uint4*>(m) = make_uint4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ void tv_st4(unsigned long long* m, const unsigned long long (&v)[4]) {
    *reinterpret_cast<ulonglong2*>(m) = make_ulonglong2(v[0], v[1]);
    *reinterpret_cast<ulonglong2*>(m + 2) = make_ulonglong2(v[2], v[3]);
}
__device__ __forceinline__ void tv_ld4(const uint32_t* m, uint32_t (&v)[4]) {
    const uint4 a = *reinterpret_cast<const uint4*>(m);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}
__device__ __forceinline__ void tv_ld4(const unsigned long long* m, unsigned long long (&v)[4]) {
    const ulonglong2 a = *reinterpret_cast<const ulonglong2*>(m), b = *reinterpret_cast<const ulonglong2*>(m + 2);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ int tv_ffs(uint32_t m) { return __ffs((int)m) - 1; }
__device__ __forceinline__ int tv_ffs(unsigned long long m) { return __ffsll((long long)m) - 1; }

// Scratch position of the tile's `nb` records (thread 0; the caller synchronises the CTA afterwards and reads *out0:
// 0xffffffff = the scratch list is full, the host grows it and reruns the batch).  Every tile records its count.
__device__ __forceinline__ void tv_place(const TvArgs& A, uint32_t t, uint32_t nb, uint32_t* out0) {
    const uint32_t at = nb ? atomicAdd(A.cursor, nb) : 0u;
    A.tile_cnt[t] = nb;
    A.tile_at[t] = at;
    if (at + nb > A.scratch_cap) {
        atomicOr(A.flags, TV_FLAG_SPACE);
        *out0 = 0xffffffffu;
    } else {
        *out0 = at;
    }
}
// range of combined-grid cells touched (the merge packs its sort keys into it)
__device__ __forceinline__ void tv_cellbb(const TvArgs& A, const int* cmin, const int* cmax, int tid) {
    if (tid < 6) {
        int* gb = A.cellbb + tid;
        const int v = tid < 3 ? cmin[tid] : cmax[tid - 3];
        if (tid < 3) { if (v < *reinterpret_cast<volatile int*>(gb)) atomicMin(gb, v); }
        else { if (v > *reinterpret_cast<volatile int*>(gb)) atomicMax(gb, v); }
    }
}

// Exclusive scan of one value per thread over the tile's CTA (kTvThreads threads).  `sm` is 34 words of shared memory.  Ends with a
// barrier so `sm` may be reused immediately.
__device__ __forceinline__ uint32_t tv_block_excl_scan(uint32_t v, uint32_t* sm, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < kTvWarps ? sm[lane] : 0u, winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(kFull, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < kTvWarps) sm[lane] = winc - w;
        if (lane == kTvWarps - 1) sm[33] = winc;
    }
    __syncthreads();
    total = sm[33];
    const uint32_t r = sm[warp] + inc - v;
    __syncthreads();
    return r;
}

template <int DT, int R>
__global__ void __launch_bounds__(kTvThreads, tv_ctas_per_sm<R>()) k_tv(AParams P, TvArgs A) {
    wait_prior();
    typedef TvGeom<R> G;
    typedef typename TvMask<R>::type M;
    extern __shared__ __align__(16) unsigned char tv_smem_raw[];
    uint16_t* const SH = reinterpret_cast<uint16_t*>(tv_smem_raw);       // planes: hash (16-bit), x, y, z, rgb
    float* const SX = reinterpret_cast<float*>(tv_smem_raw + (size_t)G::N * 2);
    float* const SY = SX + G::N;
    float* const SZ = SY + G::N;
    uint32_t* const SC = reinterpret_cast<uint32_t*>(SZ + G::N);
    float4* const items = reinterpret_cast<float4*>(tv_smem_raw);      // phase C: the tile's centroids in cell order (aliases the planes)
    constexpr int NB = TvBins<R>::value;
    typedef TvTail<NB, (int)sizeof(M)> Tail;
    Tail& S = *reinterpret_cast<Tail*>(tv_smem_raw + G::plane_bytes);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;

    if (tid == 0) { S.ticket = atomicAdd(A.ticket, 1u); S.any_valid = 0u; S.bad = 0u; }
    if (tid < 3) { S.cmin[tid] = 0x7fffffff; S.cmax[tid] = (int)0x80000000; S.bb[tid] = 0xffffffffu; S.bb[3 + tid] = 0u; }
    if (P.use_lut && tid < 256) { S.u.lut.rl[tid] = P.lut_r[tid]; S.u.lut.zl[tid] = P.lut_z[tid]; }
    if (R > 0 && tid < TvLater<R ? R : 1>::N) S.off[tid] = (uint16_t)TvLater<R ? R : 1>::offset(tid, G::NC);
    __syncthreads();
    const uint32_t t = S.ticket;
    const uint32_t per_frame = (uint32_t)(A.ntx * A.nty), nt = per_frame * (uint32_t)A.n_frames;
    if (t >= nt) return;   // (uniform; the grid is exactly nt CTAs)
    const int f = (int)(t / per_frame);
    const int rem = (int)(t - (uint32_t)f * per_frame);
    const int tyi = rem / A.ntx, txi = rem - tyi * A.ntx;
    const FrameDev& F = A.frames[f];
    const bool pass = A.frame_pass[f] != 0;
    const int y_org = P.bb + tyi * kTvH - G::HY, x_org = P.x0 + txi * kTvW - G::HX;

    float4 cen[kTvQ * 4];
    uint32_t cvalid = 0;
    int cmn[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff}, cmx[3] = {(int)0x80000000, (int)0x80000000, (int)0x80000000};
    // ---- A: evaluate core + halo into the planes (R == 0, every frame a PCL pass-through: no window, no planes — the thread's
    //      own eight pixels stay in registers as the per-frame "voxels" they are)
    {
        float fmn[3] = {INFINITY, INFINITY, INFINITY}, fmx[3] = {-INFINITY, -INFINITY, -INFINITY};
        bool over = false, anyv = false;
        if (R == 0) {
#pragma unroll
            for (int q = 0; q < kTvQ; ++q) {
                const int g = tid + q * kTvThreads;
                const int cr = g / kTvGroupsRow, cg = g - cr * kTvGroupsRow;
                const int y = y_org + cr, xb = x_org + cg * 4;
                if (y < P.bb + P.ny && xb < P.x0 + P.nx) {
                    float X[4], Y[4], Z[4];
                    const uint32_t mask = tv_eval4<DT>(P, F, S.u.lut.rl, S.u.lut.zl, xb, y, A, X, Y, Z, over);
                    if (mask) {
                        const uint32_t* c = reinterpret_cast<const uint32_t*>(F.bgr + (size_t)y * F.bgr_step + 3 * (size_t)xb);
                        const uint32_t w0 = __ldg(c), w1 = __ldg(c + 1), w2 = __ldg(c + 2);
                        const uint32_t rgb[4] = {w0 & 0x00ffffffu, (w0 >> 24) | ((w1 & 0xffffu) << 8), (w1 >> 16) | ((w2 & 0xffu) << 16),
                                                 w2 >> 8};
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (mask & (1u << j)) {
                                float4 p;
                                xform(F.T, X[j], Y[j], Z[j], p.x, p.y, p.z);
                                p.w = __uint_as_float(rgb[j]);
                                fmn[0] = fminf(fmn[0], p.x); fmx[0] = fmaxf(fmx[0], p.x);
                                fmn[1] = fminf(fmn[1], p.y); fmx[1] = fmaxf(fmx[1], p.y);
                                fmn[2] = fminf(fmn[2], p.z); fmx[2] = fmaxf(fmx[2], p.z);
                                anyv = true;
                                if (A.dbg_vox) A.dbg_vox[atomicAdd(A.dbg_cnt, 1u)] = p;   // PCL: output = *input_
                                p.z = __fadd_rn(p.z, 500.0f);   // pose_functions.cpp:1666
                                const int vi = __float2int_rd(__fmul_rn(p.x, A.icx)), vj = __float2int_rd(__fmul_rn(p.y, A.icx)),
                                          vk = __float2int_rd(__fmul_rn(p.z, A.icz));
                                cmn[0] = min(cmn[0], vi); cmx[0] = max(cmx[0], vi);
                                cmn[1] = min(cmn[1], vj); cmx[1] = max(cmx[1], vj);
                                cmn[2] = min(cmn[2], vk); cmx[2] = max(cmx[2], vk);
                                cen[q * 4 + j] = p;
                                cvalid |= 1u << (q * 4 + j);
                            }
                    }
                }
            }
        } else {
        // (the colour words are loaded whether or not a pixel turns out valid: they are in flight together with the disparity
        //  word instead of behind it — a tile's latency, not its throughput, is what costs.  Unrolling the rounds, or keeping the
        //  frame descriptor in registers, measured no better / worse: spills)
        constexpr int kRounds = (G::NG + kTvThreads - 1) / kTvThreads;
#pragma unroll 1
        for (int it = 0; it < kRounds; ++it) {
            const int g = tid + it * kTvThreads;
            if (g >= G::NG) break;
            const int lr = g / (G::NC / 4), lc = (g - lr * (G::NC / 4)) * 4;
            const int y = y_org + lr, xb = x_org + lc;
            uint2 hh = make_uint2(0xffffffffu, 0xffffffffu);
            float px[4] = {0.f, 0.f, 0.f, 0.f}, py[4] = {0.f, 0.f, 0.f, 0.f}, pz[4] = {0.f, 0.f, 0.f, 0.f};
            uint32_t rgb[4] = {0u, 0u, 0u, 0u};
            if (y >= P.bb && y < P.bb + P.ny && xb >= P.x0 && xb < P.x0 + P.nx) {   // nx % 4 == 0: a group is inside or outside
                float X[4], Y[4], Z[4];
                const uint32_t* c = reinterpret_cast<const uint32_t*>(F.bgr + (size_t)y * F.bgr_step + 3 * (size_t)xb);
                const uint32_t w0 = __ldg(c), w1 = __ldg(c + 1), w2 = __ldg(c + 2);
                const uint32_t mask = tv_eval4<DT>(P, F, S.u.lut.rl, S.u.lut.zl, xb, y, A, X, Y, Z, over);
                if (mask) {
                    rgb[0] = w0 & 0x00ffffffu;
                    rgb[1] = (w0 >> 24) | ((w1 & 0xffffu) << 8);
                    rgb[2] = (w1 >> 16) | ((w2 & 0xffu) << 16);
                    rgb[3] = w2 >> 8;
                    const bool core = lr >= G::HY && lr < G::HY + kTvH && lc >= G::HX && lc < G::HX + kTvW;
                    uint32_t h[4] = {kTvNoHash, kTvNoHash, kTvNoHash, kTvNoHash};
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (mask & (1u << j)) {
                            xform(F.T, X[j], Y[j], Z[j], px[j], py[j], pz[j]);
                            int ci, cj, ck;
                            bk_cell(px[j], py[j], pz[j], A.inv_f, ci, cj, ck);
                            h[j] = tv_hash(ci, cj, ck);
                            if (core) {
                                fmn[0] = fminf(fmn[0], px[j]); fmx[0] = fmaxf(fmx[0], px[j]);
                                fmn[1] = fminf(fmn[1], py[j]); fmx[1] = fmaxf(fmx[1], py[j]);
                                fmn[2] = fminf(fmn[2], pz[j]); fmx[2] = fmaxf(fmx[2], pz[j]);
                                anyv = true;
                            }
                        }
                    hh = make_uint2(h[0] | (h[1] << 16), h[2] | (h[3] << 16));
                }
            }
            const int o = lr * G::NC + lc;
            *reinterpret_cast<uint2*>(SH + o) = hh;
            *reinterpret_cast<float4*>(SX + o) = make_float4(px[0], px[1], px[2], px[3]);
            *reinterpret_cast<float4*>(SY + o) = make_float4(py[0], py[1], py[2], py[3]);
            *reinterpret_cast<float4*>(SZ + o) = make_float4(pz[0], pz[1], pz[2], pz[3]);
            *reinterpret_cast<uint4*>(SC + o) = make_uint4(rgb[0], rgb[1], rgb[2], rgb[3]);
        }
        }
        // the frame's exact bbox (PCL getMinMax3D) from the core pixels: every pixel is core in exactly one tile
        const unsigned anyw = __ballot_sync(kFull, anyv);
        if (anyw) {
            uint32_t mn[3], mx[3];   // (order-preserving uint images: -0 < +0 as in the other engines' integer reductions)
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                mn[a] = __reduce_min_sync(kFull, anyv ? f2ord(fmn[a]) : 0xffffffffu);
                mx[a] = __reduce_max_sync(kFull, anyv ? f2ord(fmx[a]) : 0u);
            }
            if (lane == 0) {
                S.any_valid = 1u;
#pragma unroll
                for (int a = 0; a < 3; ++a) { atomicMin(&S.bb[a], mn[a]); atomicMax(&S.bb[3 + a], mx[a]); }
            }
        }
        if (over && !pass) S.bad = 1u;   // (a pass-through frame has no window to break)
    }
    __syncthreads();
    if (S.any_valid && tid < 6) {
        uint32_t* gb = A.bbox + (size_t)f * 6 + tid;
        const uint32_t v = S.bb[tid];
        if (tid < 3) { if (v < *reinterpret_cast<volatile uint32_t*>(gb)) atomicMin(gb, v); }
        else { if (v > *reinterpret_cast<volatile uint32_t*>(gb)) atomicMax(gb, v); }
    }
    if (tid == 0 && S.bad) atomicOr(A.flags, TV_FLAG_RANGE);

    // ---- B: the leaves.  A pixel's leaf-mates lie in its window; it is its leaf's FIRST point iff no earlier pixel marks it.
    if (R > 0 && !pass) {
        typedef TvLater<R> LW;
        M* const mlS = reinterpret_cast<M*>(&S.u);   // (the LUT is dead, the cell counters not yet alive) per core pixel: its verified later mates
        // B1  every pixel of the core and of the halo rows above / columns beside it compares the hashes of the window positions
        //     LATER in scan order (half of the window: every pair is looked at once), verifies an equal hash on the cell itself,
        //     and marks the mate "not first" (bit 31 of its colour word: all writers write the same value).  Core pixels keep
        //     the mask of their verified mates.
        for (int g = tid; g < (G::HY + kTvH) * (G::NC / 4); g += kTvThreads) {
            const int lr = g / (G::NC / 4), lc = (g - lr * (G::NC / 4)) * 4;
            const int o = lr * G::NC + lc;
            const uint2 h2 = *reinterpret_cast<const uint2*>(SH + o);
            if ((h2.x & h2.y) == 0xffffffffu) {   // nothing valid here (masks of a core group: none)
                if (lr >= G::HY && lc >= G::HX && lc < G::HX + kTvW) {
                    const M zero[4] = {0, 0, 0, 0};
                    tv_st4(mlS + ((lr - G::HY) * kTvW + (lc - G::HX)), zero);
                }
                continue;
            }
            const uint32_t h[4] = {h2.x & 0xffffu, h2.x >> 16, h2.y & 0xffffu, h2.y >> 16};
            M ml[4] = {0, 0, 0, 0};
            const uint2 none = make_uint2(0xffffffffu, 0xffffffffu);
#pragma unroll
            for (int dr = 0; dr <= R; ++dr) {
                const uint16_t* hr = SH + (lr + dr) * G::NC + lc - 4;
                const uint2 a = (lc >= 4 && dr > 0) ? *reinterpret_cast<const uint2*>(hr) : none;
                const uint2 b = *reinterpret_cast<const uint2*>(hr + 4);
                const uint2 c = (lc + 8 <= G::NC) ? *reinterpret_cast<const uint2*>(hr + 8) : none;
                const uint32_t w[12] = {a.x & 0xffffu, a.x >> 16, a.y & 0xffffu, a.y >> 16, b.x & 0xffffu, b.x >> 16,
                                        b.y & 0xffffu, b.y >> 16, c.x & 0xffffu, c.x >> 16, c.y & 0xffffu, c.y >> 16};
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int dc = (dr == 0 ? 1 : -R); dc <= R; ++dc)
                        if (w[4 + j + dc] == h[j]) ml[j] |= (M)1 << LW::bit(dr, dc);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                M l = h[j] == kTvNoHash ? (M)0 : ml[j], keep = 0;
                if (l) {
                    const int oc = o + j;
                    int ci, cj, ck;
                    bk_cell(SX[oc], SY[oc], SZ[oc], A.inv_f, ci, cj, ck);
                    while (l) {
                        const int k = tv_ffs(l);
                        l &= l - 1;
                        const int on = oc + (int)S.off[k];
                        int ni, nj, nk;
                        bk_cell(SX[on], SY[on], SZ[on], A.inv_f, ni, nj, nk);
                        if (ni == ci && nj == cj && nk == ck) {
                            keep |= (M)1 << k;
                            SC[on] |= 0x80000000u;
                        }
                    }
                }
                ml[j] = keep;
            }
            if (lr >= G::HY && lc >= G::HX && lc < G::HX + kTvW) tv_st4(mlS + ((lr - G::HY) * kTvW + (lc - G::HX)), ml);
        }
        __syncthreads();
        // B2  a first point with mates left-folds them in scan order — the oracle's stable order, so the per-frame VoxelGrid
        //     centroid is bit-identical — divides (pcl::CentroidPoint) and leaves the centroid in its own plane slot (nobody else
        //     reads a first point any more).  Each lane walks its own pending pixels back to back.
        uint32_t todo = 0;
#pragma unroll
        for (int q = 0; q < kTvQ; ++q) {
            const int g = tid + q * kTvThreads;
            const int o = (g / kTvGroupsRow + G::HY) * G::NC + (g % kTvGroupsRow) * 4 + G::HX;
            const uint2 h2 = *reinterpret_cast<const uint2*>(SH + o);
            const uint4 c4 = *reinterpret_cast<const uint4*>(SC + o);
            const uint32_t hv[4] = {h2.x & 0xffffu, h2.x >> 16, h2.y & 0xffffu, h2.y >> 16}, cv[4] = {c4.x, c4.y, c4.z, c4.w};
            M mv[4];
            tv_ld4(mlS + g * 4, mv);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (hv[j] != kTvNoHash && !(cv[j] & 0x80000000u) && mv[j] != 0) todo |= 1u << (q * 4 + j);
        }
        while (todo) {
            const int r = __ffs((int)todo) - 1;
            todo &= todo - 1;
            const int g = tid + (r >> 2) * kTvThreads;
            const int oc = (g / kTvGroupsRow + G::HY) * G::NC + (g % kTvGroupsRow) * 4 + G::HX + (r & 3);
            M l = mlS[g * 4 + (r & 3)];
            float sx = __fadd_rn(0.f, SX[oc]), sy = __fadd_rn(0.f, SY[oc]), sz = __fadd_rn(0.f, SZ[oc]);   // (the oracle's sums start at +0)
            uint32_t w = SC[oc];
            uint32_t cn = 1, cr = (w >> 16) & 255u, cg = (w >> 8) & 255u, cb = w & 255u;
            while (l) {
                const int k = tv_ffs(l);
                l &= l - 1;
                const int on = oc + (int)S.off[k];
                sx = __fadd_rn(sx, SX[on]); sy = __fadd_rn(sy, SY[on]); sz = __fadd_rn(sz, SZ[on]);
                w = SC[on];
                cr += (w >> 16) & 255u; cg += (w >> 8) & 255u; cb += w & 255u;
                ++cn;
            }
            const float4 c = bk_centroid(sx, sy, sz, cn, cr, cg, cb);
            SX[oc] = c.x; SY[oc] = c.y; SZ[oc] = c.z; SC[oc] = __float_as_uint(c.w);
        }
        __syncthreads();
    }
    if (R > 0) {   // the thread's own core pixels: the unmarked ones are the per-frame voxels
#pragma unroll
        for (int r = 0; r < kTvQ * 4; ++r) {
            const int g = tid + (r >> 2) * kTvThreads;
            const int o = (g / kTvGroupsRow + G::HY) * G::NC + (g % kTvGroupsRow) * 4 + G::HX;
            // (16-byte loads of the group's four pixels; the compiler keeps one copy per group)
            const uint2 h2 = *reinterpret_cast<const uint2*>(SH + o);
            const uint4 c4 = *reinterpret_cast<const uint4*>(SC + o);
            const float4 x4 = *reinterpret_cast<const float4*>(SX + o), y4 = *reinterpret_cast<const float4*>(SY + o),
                         z4 = *reinterpret_cast<const float4*>(SZ + o);
            const int j = r & 3;
            const uint32_t hq = j == 0 ? (h2.x & 0xffffu) : j == 1 ? (h2.x >> 16) : j == 2 ? (h2.y & 0xffffu) : (h2.y >> 16);
            const uint32_t w = j == 0 ? c4.x : j == 1 ? c4.y : j == 2 ? c4.z : c4.w;
            if (hq == kTvNoHash || (w & 0x80000000u)) continue;
            float4 c = make_float4(j == 0 ? x4.x : j == 1 ? x4.y : j == 2 ? x4.z : x4.w, j == 0 ? y4.x : j == 1 ? y4.y : j == 2 ? y4.z : y4.w,
                                   j == 0 ? z4.x : j == 1 ? z4.y : j == 2 ? z4.z : z4.w, __uint_as_float(w));
            if (!pass) {   // a leaf of one point: (0 + x) / 1 — only -0 changes, to +0 (a folded centroid is never -0); PCL's
                           // pass-through keeps the point as it is
                c.x = __fadd_rn(0.f, c.x); c.y = __fadd_rn(0.f, c.y); c.z = __fadd_rn(0.f, c.z);
            }
            if (A.dbg_vox) A.dbg_vox[atomicAdd(A.dbg_cnt, 1u)] = c;
            c.z = __fadd_rn(c.z, 500.0f);   // pose_functions.cpp:1666
            const int vi = __float2int_rd(__fmul_rn(c.x, A.icx)), vj = __float2int_rd(__fmul_rn(c.y, A.icx)),
                      vk = __float2int_rd(__fmul_rn(c.z, A.icz));
            cmn[0] = min(cmn[0], vi); cmx[0] = max(cmx[0], vi);
            cmn[1] = min(cmn[1], vj); cmx[1] = max(cmx[1], vj);
            cmn[2] = min(cmn[2], vk); cmx[2] = max(cmx[2], vk);
            cen[r] = c;
            cvalid |= 1u << r;
        }
    }
    // ---- C: the tile's cells -------------------------------------------------------------------------------------------
    {
        const unsigned anyc = __ballot_sync(kFull, cvalid != 0u);
        if (anyc) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                cmn[a] = __reduce_min_sync(kFull, cmn[a]);
                cmx[a] = __reduce_max_sync(kFull, cmx[a]);
            }
            if (lane == 0) {
#pragma unroll
                for (int a = 0; a < 3; ++a) { atomicMin(&S.cmin[a], cmn[a]); atomicMax(&S.cmax[a], cmx[a]); }
            }
        }
    }
    __syncthreads();   // (the planes are dead from here on; the LUT as well)
    const bool have = S.cmin[0] != 0x7fffffff;
    const int c0i = S.cmin[0], c0j = S.cmin[1], c0k = S.cmin[2];
    const long long ei = have ? (long long)S.cmax[0] - c0i + 1 : 0, ej = have ? (long long)S.cmax[1] - c0j + 1 : 0,
                    ek = have ? (long long)S.cmax[2] - c0k + 1 : 0;
    const bool fits = ei * ej * ek <= (long long)NB && ei <= NB && ej <= NB && ek <= NB;
    int nbins = fits ? (int)(ei * ej * ek) : 0;
    const int Bi = 1 << 20;
    uint32_t bin[kTvQ * 4], rk[kTvQ * 4];   // cell number of the thread's centroids (NB + 1: none), rank inside the cell
#pragma unroll
    for (int r = 0; r < kTvQ * 4; ++r) bin[r] = (uint32_t)(NB + 1);
    bool loose = false;
    if (fits) {   // the box of the tile's cells indexes the table directly
#pragma unroll
        for (int r = 0; r < kTvQ * 4; ++r)
            if ((cvalid >> r) & 1u) {
                const int vi = __float2int_rd(__fmul_rn(cen[r].x, A.icx)), vj = __float2int_rd(__fmul_rn(cen[r].y, A.icx)),
                          vk = __float2int_rd(__fmul_rn(cen[r].z, A.icz));
                bin[r] = (uint32_t)(((vk - c0k) * (int)ej + (vj - c0j)) * (int)ei + (vi - c0i));
            }
    } else {
        // The cells span more than the table (a depth discontinuity inside the tile, a combined grid that is fine against the
        // sideways scatter of noisy depths): number the cells that are actually occupied through an open-addressing hash of the
        // 64-bit cell key.  Which number a cell gets depends on a race, i.e. only the order of DIFFERENT cells' records does.
        unsigned long long* const tab = reinterpret_cast<unsigned long long*>(tv_smem_raw);
        uint16_t* const dense = reinterpret_cast<uint16_t*>(tv_smem_raw + (size_t)kTvHash * 8);
        {
            uint4* tz = reinterpret_cast<uint4*>(tab);
            for (int i = tid; i < kTvHash / 2; i += kTvThreads) tz[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
            if (tid == 0) S.nbh = 0u;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < kTvQ * 4; ++r)
            if ((cvalid >> r) & 1u) {
                const int vi = __float2int_rd(__fmul_rn(cen[r].x, A.icx)), vj = __float2int_rd(__fmul_rn(cen[r].y, A.icx)),
                          vk = __float2int_rd(__fmul_rn(cen[r].z, A.icz));
                const unsigned long long k = ((unsigned long long)(uint32_t)(vk + Bi) << 42) | ((unsigned long long)(uint32_t)(vj + Bi) << 21) |
                                             (unsigned long long)(uint32_t)(vi + Bi);
                uint32_t h = ((uint32_t)(k ^ (k >> 21) ^ (k >> 42)) * 0x9e3779b1u) >> kTvHashShift;
                for (;;) {
                    const unsigned long long old = atomicCAS(&tab[h], ~0ull, k);
                    if (old == ~0ull) { dense[h] = (uint16_t)atomicAdd(&S.nbh, 1u); break; }
                    if (old == k) break;
                    h = (h + 1) & (kTvHash - 1);
                }
                bin[r] = h;
            }
        __syncthreads();
        nbins = (int)S.nbh;
        loose = nbins > NB;
        if (!loose) {
#pragma unroll
            for (int r = 0; r < kTvQ * 4; ++r)
                if ((cvalid >> r) & 1u) bin[r] = dense[bin[r]];
        }
        __syncthreads();   // (the table is dead: the centroids in cell order take its place)
    }
    if (loose) {
        // more occupied cells than the table numbers (at least every second centroid alone in its cell): every centroid leaves
        // as its own single-point record, in tile order (thread, slot)
        uint32_t tot;
        uint32_t pos = tv_block_excl_scan((uint32_t)__popc(cvalid), S.scan, tot);
        if (tid == 0) tv_place(A, t, tot, &S.out0);
        __syncthreads();
        if (tot == 0) return;
        if (tid == 0) atomicAdd(A.frame_vox + f, tot);
        tv_cellbb(A, S.cmin, S.cmax, tid);
        if (S.out0 == 0xffffffffu) return;
        o3r_cell* const out = A.scratch + S.out0;
#pragma unroll
        for (int r = 0; r < kTvQ * 4; ++r)
            if ((cvalid >> r) & 1u) {
                const float4 p = cen[r];
                const int vi = __float2int_rd(__fmul_rn(p.x, A.icx)), vj = __float2int_rd(__fmul_rn(p.y, A.icx)),
                          vk = __float2int_rd(__fmul_rn(p.z, A.icz));
                const uint32_t w = __float_as_uint(p.w);
                o3r_cell c;
                c.key = ((unsigned long long)(uint32_t)(vk + Bi) << 42) | ((unsigned long long)(uint32_t)(vj + Bi) << 21) |
                        (unsigned long long)(uint32_t)(vi + Bi);
                c.sx = p.x; c.sy = p.y; c.sz = p.z; c.n = 1u;
                c.sr = (w >> 16) & 255u; c.sg = (w >> 8) & 255u; c.sb = w & 255u; c.pad = 0u;
                out[pos++] = c;
            }
        return;
    }
    for (int b = tid; b < (nbins + 2) * kTvWarps; b += kTvThreads) {
        const int w = b / (nbins + 2), i = b - w * (nbins + 2);
        S.u.cnt[w][i == nbins + 1 ? NB + 1 : i] = 0;
    }
    __syncthreads();
    // stable rank of every centroid inside its cell (tile order = warp, slot, lane); lanes without a centroid share the
    // stand-in cell NB + 1
    uint16_t* wc = &S.u.cnt[warp][0];
#pragma unroll
    for (int r = 0; r < kTvQ * 4; ++r) {
        const unsigned peers = __match_any_sync(kFull, bin[r]);
        const uint32_t old = wc[bin[r]];
        __syncwarp();
        if ((peers & lt) == 0u) wc[bin[r]] = (uint16_t)(old + __popc(peers));
        __syncwarp();
        rk[r] = old + __popc(peers & lt);
    }
    __syncthreads();
    // per cell: exclusive prefix over the warps; then first item / rank among the non-empty cells (packed scan)
    {
        constexpr int BPT = NB / kTvThreads;   // cells per thread
        uint32_t run[BPT], psum = 0;
#pragma unroll
        for (int qq = 0; qq < BPT; ++qq) {
            const int b = tid * BPT + qq;
            uint32_t acc = 0;
            if (b < nbins) {
#pragma unroll
                for (int w = 0; w < kTvWarps; ++w) { const uint32_t c = S.u.cnt[w][b]; S.u.cnt[w][b] = (uint16_t)acc; acc += c; }
            }
            run[qq] = acc | (acc ? 1u << 16 : 0u);
            psum += run[qq];
        }
        uint32_t tot;
        uint32_t ds = tv_block_excl_scan(psum, S.scan, tot);
#pragma unroll
        for (int qq = 0; qq < BPT; ++qq) {
            const int b = tid * BPT + qq;
            if (b < nbins) S.bd[b] = ds;
            ds += run[qq];
        }
        if (tid == 0) { S.bd[nbins] = tot; S.nitems = tot & 0xffffu; S.nb = tot >> 16; }
    }
    __syncthreads();
    const uint32_t nb = S.nb;
#pragma unroll
    for (int r = 0; r < kTvQ * 4; ++r)
        if ((cvalid >> r) & 1u) items[(S.bd[bin[r]] & 0xffffu) + (uint32_t)wc[bin[r]] + rk[r]] = cen[r];
    if (tid == 0) tv_place(A, t, nb, &S.out0);
    __syncthreads();
    if (nb == 0) return;
    if (tid == 0) atomicAdd(A.frame_vox + f, S.nitems);
    tv_cellbb(A, S.cmin, S.cmax, tid);
    if (S.out0 == 0xffffffffu) return;
    o3r_cell* const out = A.scratch + S.out0;
    // four lanes per cell: lane s left-folds items s, s + 4, ... of the cell, then (s0 + s1) + (s2 + s3): a fixed tree
    for (int b0 = warp * 8; b0 < nbins; b0 += kTvWarps * 8) {
        const int b = b0 + (lane >> 2), sub = lane & 3;
        uint32_t a = 0, e = 0, dense = 0;
        if (b < nbins) {
            const uint32_t v0 = S.bd[b], v1 = S.bd[b + 1];
            a = v0 & 0xffffu; e = v1 & 0xffffu; dense = v0 >> 16;
        }
        float sx = 0.f, sy = 0.f, sz = 0.f;
        uint32_t cr = 0, cg = 0, cb = 0;
        for (uint32_t i = a + sub; i < e; i += 4) {
            const float4 p = items[i];
            sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z);
            const uint32_t w = __float_as_uint(p.w);
            cr += (w >> 16) & 255u; cg += (w >> 8) & 255u; cb += w & 255u;
        }
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
            sx = __fadd_rn(sx, __shfl_xor_sync(kFull, sx, o));
            sy = __fadd_rn(sy, __shfl_xor_sync(kFull, sy, o));
            sz = __fadd_rn(sz, __shfl_xor_sync(kFull, sz, o));
            cr += __shfl_xor_sync(kFull, cr, o); cg += __shfl_xor_sync(kFull, cg, o); cb += __shfl_xor_sync(kFull, cb, o);
        }
        if (sub == 0 && e > a) {
            const float4 p0 = items[a];
            const int vi = __float2int_rd(__fmul_rn(p0.x, A.icx)), vj = __float2int_rd(__fmul_rn(p0.y, A.icx)),
                      vk = __float2int_rd(__fmul_rn(p0.z, A.icz));
            o3r_cell c;
            c.key = ((unsigned long long)(uint32_t)(vk + Bi) << 42) | ((unsigned long long)(uint32_t)(vj + Bi) << 21) |
                    (unsigned long long)(uint32_t)(vi + Bi);
            c.sx = sx; c.sy = sy; c.sz = sz; c.n = e - a;
            c.sr = cr; c.sg = cg; c.sb = cb; c.pad = 0u;
            out[dense] = c;
        }
    }
}

// The chunk's records in tile order: one warp per tile copies its records from the scratch list to
// out[*out_base + tile_off[t] ...) (tile_off = exclusive scan of tile_cnt, *chunk_total its total).  40-byte records move as
// five 8-byte words.  The list is skipped (TV_FLAG_SPACE) when the scratch list overflowed or the output would.
__global__ void __launch_bounds__(kThreads) k_tv_compact(const o3r_cell* __restrict__ scratch, const uint32_t* __restrict__ tile_cnt,
                                                         const uint32_t* __restrict__ tile_at, const uint32_t* __restrict__ tile_off,
                                                         uint32_t n_tiles, o3r_cell* __restrict__ out,
                                                         const uint32_t* __restrict__ out_base, const uint32_t* __restrict__ chunk_total,
                                                         uint32_t out_cap, const uint32_t* __restrict__ cursor,
                                                         uint32_t* __restrict__ max_cursor, uint32_t* __restrict__ flags, int n_frames,
                                                         const uint32_t* __restrict__ bbox, float inv_f,
                                                         const uint8_t* __restrict__ guess, uint8_t* __restrict__ actual) {
    wait_prior();
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicMax(max_cursor, *cursor);
    // per frame: PCL's int32 overflow guard on the exact bbox against the guess the tile kernel ran on
    if (blockIdx.x == gridDim.x - 1)
        for (int f = threadIdx.x; f < n_frames; f += kThreads) {
            const GridParams G = make_grid(bbox + 6 * f, inv_f, inv_f, inv_f);
            const uint8_t a = (uint8_t)(G.passthrough ? 1 : 0);
            actual[f] = G.empty ? guess[f] : a;   // a frame without points has nothing to get wrong
            if (!G.empty && a != guess[f]) atomicOr(flags, TV_FLAG_PASS);
        }
    const bool room = (unsigned long long)*out_base + *chunk_total <= (unsigned long long)out_cap;
    if (!room && blockIdx.x == 0 && threadIdx.x == 0) atomicOr(flags, TV_FLAG_SPACE);
    if (!room || (*flags & TV_FLAG_SPACE)) return;
    const uint32_t t = blockIdx.x * kWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (t >= n_tiles) return;
    const uint32_t n = tile_cnt[t];
    if (n == 0) return;
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(scratch + tile_at[t]);
    unsigned long long* dst = reinterpret_cast<unsigned long long*>(out + *out_base + tile_off[t]);
    const uint32_t nw = n * 5u;
    uint32_t i = lane;
    for (; i + 96u < nw; i += 128u) {   // four independent loads in flight per lane
        const unsigned long long a = __ldcs(src + i), b = __ldcs(src + i + 32), c = __ldcs(src + i + 64), d = __ldcs(src + i + 96);
        dst[i] = a; dst[i + 32] = b; dst[i + 64] = c; dst[i + 96] = d;
    }
    for (; i < nw; i += 32u) dst[i] = __ldcs(src + i);
}

}  // namespace o3r
