// bucket.cuh — the fused disparity -> cloud -> voxel engine (O3R_MERGE_ACCUMULATE_FUSED).
//
// What it replaces: createSingleImgPtCloud (pose_functions.cpp:1030-1134) + transformPtCloud (:1358-1362) +
// downsamplePtCloud(cloud, false) (:1654-1709, VoxelGrid leaf voxel_size / 5) + the append to cloud_big (pose.cpp:434)
// of a whole cycle, up to the partial sums the incremental merge (voxel.cuh engine 2) folds into the resident shard.
//
// Why not the radix sort of engine 1: PCL sorts the whole frame by leaf index only to GROUP the points of a leaf; a
// sort-based VoxelGrid moves ~110 B per point through HBM where 20 B are compulsory.  A leaf of voxel_size / 5 only holds
// points that are a few pixels apart, so the grouping is local: the cycle's points are binned ONCE into buckets of
// kBkB x kBkB leaf columns (all z) — nominally one combined-grid (voxel_size, voxel_size, 1000) cell — and each bucket
// (~80 points at 720p, voxel_size 0.05) is finished inside shared memory by one warp:
//
//   k_bk_hist     every pixel: validity, reprojection, transform -> leaf cell -> bucket; counts per bucket (RED), the
//                 frame's PCL bbox (for the int32 overflow guard)
//   k_bk_scan     exclusive scan of the bucket counts (decoupled look-back) + compact list of the non-empty buckets
//   k_bk_scatter  the same evaluation again + colour; the tile's points are staged in shared memory in scan order, every
//                 run of consecutive points of one bucket reserves its slots with ONE atomic, and the records leave as
//                 coalesced bursts: {x, y, z, rgb} (16 B) + scan position (4 B)
//   k_bk_reduce   one warp per bucket: counting sort by leaf column, rank inside the column by (z cell, scan position)
//                 -> the bucket in PCL's order restricted to it; every leaf is left-folded in scan order (bit-identical
//                 centroids: the oracle's stable order), each centroid is celled on the combined grid and the warp emits
//                 one partial cell per distinct combined cell (nearly always one), at an offset from a decoupled
//                 look-back so the partial list is reproducible.
//
// Determinism: the slot a point gets inside its bucket depends on an atomic race, which is why the scan position
// travels with it — the reduce orders by it, so every float is summed in a fixed order.  Leaf centroids are bit-exact;
// the combined-grid partial is a fixed tree (per lane in leaf order, then an xor butterfly), i.e. the same contract as
// O3R_MERGE_ACCUMULATE_TILED: keys, counts, colour sums exact, centroids equal to the oracle's left fold within float
// reassociation (<= 1e-5 relative), reproducible bit for bit from run to run.
//
// Limits (checked on the device; the host then reruns the batch through the sort engine and stays there): a bucket with
// more than kBkCapSlow points (histogram), or more than one reduce CTA holds (kRdCap), more than kRdStray strays in one
// bucket or more than the host's stray cap in one chunk (reduce), a point outside the host's conservative per-frame bucket
// grid.  A frame whose grid the host cannot bound (w changing sign, a cell index past 8e6 leaf edges, more than 2^24
// buckets) keeps the batch off this engine from the start.
#pragma once
#include "common.cuh"
#include "sort.cuh"
#include "stage_a.cuh"

namespace o3r {

constexpr int kBkB = 5;                            // bucket edge in leaf cells (= voxel_size / leaf)
constexpr int kBkSub = kBkB * kBkB;                // leaf columns per bucket (<= 32: one lane per column in the scan)
constexpr int kBkCapSlow = 65535;                  // points of one bucket: its count shares a 32-bit word with the frame index
constexpr int kBkScanItems = 8;
constexpr int kBkScanTile = kThreads * kBkScanItems;
#ifndef O3R_BK_MINB
#define O3R_BK_MINB 4
#endif
constexpr int kBkKBits = 26;                       // (z cell - k0) must fit: (2^26 * 25) < 2^32

// per-frame bucket grid, from the host's conservative bound of the frame's world bbox
struct BkFrame {
    int i0c, j0c;        // leaf cell of the grid origin (multiples of kBkB)
    int ni, nj;          // extent in buckets
    int k0;              // lower bound of the z leaf cell
    uint32_t base;       // first bucket of the frame in the batch-wide arrays
    int pad0, pad1;
};

enum { BK_FLAG_RANGE = 1u, BK_FLAG_BUCKET = 2u, BK_FLAG_PART = 4u };

__device__ __forceinline__ void bk_cell(float x, float y, float z, float inv, int& i, int& j, int& k) {
    i = __float2int_rd(__fmul_rn(x, inv));   // == (int)floorf(.) for every value an int holds, one conversion instead of two
    j = __float2int_rd(__fmul_rn(y, inv));
    k = __float2int_rd(__fmul_rn(z, inv));
}

// bucket of leaf column (i, j); `bad` is raised when the column lies outside the frame's grid (the index is then clamped:
// still a function of (i, j) only, and in bounds)
__device__ __forceinline__ uint32_t bk_index(const BkFrame& B, int i, int j, int k, bool& bad) {
    int bi = i - B.i0c, bj = j - B.j0c;
    const unsigned kr = (unsigned)(k - B.k0);
    if (bi < 0 || bj < 0 || kr >= (1u << kBkKBits)) { bad = true; bi = max(bi, 0); bj = max(bj, 0); }
    int I = bi / kBkB, J = bj / kBkB;
    if (I >= B.ni || J >= B.nj) { bad = true; I = min(I, B.ni - 1); J = min(J, B.nj - 1); }
    return B.base + (uint32_t)J * (uint32_t)B.ni + (uint32_t)I;
}

// ---- pass 1: bucket histogram + per-frame bbox ---------------------------------------------------------------------
template <int DT>
__global__ void __launch_bounds__(kThreads) k_bk_hist(AParams P, const FrameDev* __restrict__ frames,
                                                      const BkFrame* __restrict__ bk, float inv_f,
                                                      uint32_t* __restrict__ counts, uint32_t* __restrict__ bbox,
                                                      uint32_t* __restrict__ flags) {
    wait_prior();
    __shared__ double rl[256];
    __shared__ float zl[256];
    __shared__ uint32_t s_red[8];
    const int tile = blockIdx.x, f = blockIdx.y;
    const FrameDev& F = frames[f];
    const BkFrame B = bk[f];
    if (threadIdx.x < 8) s_red[threadIdx.x] = (threadIdx.x < 3) ? 0xffffffffu : 0u;
    load_lut(P, rl, zl);
    Samp S;
    eval4<DT>(P, F, rl, zl, tile, S);
    uint32_t mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u};
    uint32_t cur = 0xffffffffu, run = 0;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (S.mask & (1u << j)) {
            float tx, ty, tz;
            xform(F.T, S.x[j], S.y[j], S.z[j], tx, ty, tz);
            const uint32_t ox = f2ord(tx), oy = f2ord(ty), oz = f2ord(tz);
            mn[0] = min(mn[0], ox); mx[0] = max(mx[0], ox);
            mn[1] = min(mn[1], oy); mx[1] = max(mx[1], oy);
            mn[2] = min(mn[2], oz); mx[2] = max(mx[2], oz);
            int ci, cj, ck;
            bk_cell(tx, ty, tz, inv_f, ci, cj, ck);
            const uint32_t b = bk_index(B, ci, cj, ck, bad);
            if (b == cur) ++run;
            else {
                if (run) atomicAdd(&counts[cur], run);
                cur = b; run = 1;
            }
        }
    if (run) atomicAdd(&counts[cur], run);
    if (bad) atomicOr(flags, BK_FLAG_RANGE);
    const uint32_t any = __ballot_sync(kFull, S.mask != 0u);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        mn[a] = __reduce_min_sync(kFull, mn[a]);
        mx[a] = __reduce_max_sync(kFull, mx[a]);
    }
    if ((threadIdx.x & 31) == 0 && any) {
        atomicAdd(&s_red[6], 1u);
#pragma unroll
        for (int a = 0; a < 3; ++a) { atomicMin(&s_red[a], mn[a]); atomicMax(&s_red[3 + a], mx[a]); }
    }
    __syncthreads();
    if (threadIdx.x < 6 && s_red[6]) {
        if (threadIdx.x < 3) atomicMin(&bbox[f * 6 + threadIdx.x], s_red[threadIdx.x]);
        else atomicMax(&bbox[f * 6 + threadIdx.x], s_red[threadIdx.x]);
    }
}

// per frame: PCL's int32 overflow guard on the exact bbox (pass-through frames keep their points verbatim)
__global__ void k_bk_frames(int n_frames, const uint32_t* __restrict__ bbox, float inv_f, uint8_t* __restrict__ frame_pass,
                            uint32_t* __restrict__ frame_vox) {
    wait_prior();
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    const GridParams G = make_grid(bbox + 6 * f, inv_f, inv_f, inv_f);
    frame_pass[f] = (uint8_t)(G.passthrough ? 1 : 0);
    frame_vox[f] = 0u;
}

// ---- exclusive scan of the bucket counts + list of the non-empty buckets -----------------------------------------------
// status word: flag << 62 | non-empty buckets << 34 | points
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
constexpr unsigned long long kBk64Local = 1ull << 62, kBk64Global = 2ull << 62, kBk64Mask = (1ull << 62) - 1ull;

// counts[g] becomes the bucket's first slot (the scatter's cursor); nl[r] = {first slot, points | frame << 16, I, J} of the
// r-th non-empty bucket ((I, J) = the bucket's position in units of kBkB leaf cells = its nominal cell on the combined grid;
// the frame is chunk-local and takes all 16 bits: a chunk holds up to 65535 frames); totals = {points, non-empty buckets}
__global__ void __launch_bounds__(kThreads) k_bk_scan(uint32_t* __restrict__ counts, uint32_t nb_total,
                                                      const BkFrame* __restrict__ bk, int n_frames, uint4* __restrict__ nl,
                                                      unsigned long long* __restrict__ status, uint32_t* __restrict__ ticket,
                                                      uint32_t* __restrict__ totals, uint32_t* __restrict__ flags) {
    wait_prior();
    __shared__ unsigned long long s_w[kWarps + 2];
    __shared__ uint32_t s_ticket;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_ticket = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t t = s_ticket;
    const uint32_t nt = (nb_total + kBkScanTile - 1) / kBkScanTile;
    if (t >= nt) return;
    const uint32_t g0 = t * kBkScanTile + tid * kBkScanItems;
    uint32_t c[kBkScanItems];
    if (g0 + kBkScanItems <= nb_total) {
        const uint4 a = *reinterpret_cast<const uint4*>(counts + g0), b = *reinterpret_cast<const uint4*>(counts + g0 + 4);
        c[0] = a.x; c[1] = a.y; c[2] = a.z; c[3] = a.w; c[4] = b.x; c[5] = b.y; c[6] = b.z; c[7] = b.w;
    } else {
#pragma unroll
        for (int q = 0; q < kBkScanItems; ++q) c[q] = g0 + q < nb_total ? counts[g0 + q] : 0u;
    }
    unsigned long long mine = 0;
    bool over = false;
#pragma unroll
    for (int q = 0; q < kBkScanItems; ++q) {
        mine += (unsigned long long)c[q] + (c[q] ? (1ull << 34) : 0ull);
        over = over || c[q] > (uint32_t)kBkCapSlow;
    }
    if (over) atomicOr(flags, BK_FLAG_BUCKET);
    // CTA-wide exclusive scan of the packed (non-empty, points) pair
    unsigned long long inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const unsigned long long w = lane < kWarps ? s_w[lane] : 0ull;
        unsigned long long winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(kFull, winc, o);
            if (lane >= o) winc += v;
        }
        if (lane < kWarps) s_w[lane] = winc - w;
        const unsigned long long tile_tot = __shfl_sync(kFull, winc, kWarps - 1);
        // decoupled look-back over the predecessors' totals, 32 tiles per step
        if (lane == 0) st_relaxed_u64(status + t, (t == 0 ? kBk64Global : kBk64Local) | tile_tot);
        unsigned long long pf = 0;
        for (int32_t back = (int32_t)t - 1; back >= 0; back -= 32) {
            const int32_t idx = back - lane;
            unsigned long long v = kBk64Global;
            if (idx >= 0)
                while (((v = ld_relaxed_u64(status + idx)) >> 62) == 0ull) __nanosleep(32);
            const unsigned gm = __ballot_sync(kFull, (v >> 62) == 2ull);
            const int first = gm ? __ffs(gm) - 1 : 31;
            unsigned long long part = lane <= first ? (v & kBk64Mask) : 0ull;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(kFull, part, o);
            pf += part;
            if (gm) break;
        }
        if (lane == 0) {
            if (t > 0) st_relaxed_u64(status + t, kBk64Global | (pf + tile_tot));
            s_w[kWarps] = pf;
            if (t == nt - 1) {
                const unsigned long long all = pf + tile_tot;
                totals[0] = (uint32_t)(all & ((1ull << 34) - 1ull));
                totals[1] = (uint32_t)(all >> 34);
            }
        }
    }
    __syncthreads();
    unsigned long long ex = s_w[kWarps] + s_w[warp] + inc - mine;
    uint32_t start = (uint32_t)(ex & ((1ull << 34) - 1ull)), rank = (uint32_t)(ex >> 34);
    // frame of the thread's first bucket (the buckets of a frame are contiguous), advanced as g crosses a base
    int f = 0;
    if (g0 < nb_total) {
        int lo = 0, hi = n_frames - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (bk[mid].base <= g0) lo = mid; else hi = mid - 1;
        }
        f = lo;
    }
    uint32_t next_base = (f + 1 < n_frames) ? bk[f + 1].base : 0xffffffffu;
    uint32_t o[kBkScanItems];
#pragma unroll
    for (int q = 0; q < kBkScanItems; ++q) {
        const uint32_t g = g0 + q;
        o[q] = start;
        if (g < nb_total && c[q]) {
            while (g >= next_base) { ++f; next_base = (f + 1 < n_frames) ? bk[f + 1].base : 0xffffffffu; }
            const BkFrame Bf = bk[f];
            const uint32_t lg = g - Bf.base;
            const int nI = Bf.i0c / kBkB + (int)(lg % (uint32_t)Bf.ni), nJ = Bf.j0c / kBkB + (int)(lg / (uint32_t)Bf.ni);
            nl[rank++] = make_uint4(start, min(c[q], 0xffffu) | ((uint32_t)f << 16), (uint32_t)nI, (uint32_t)nJ);
            start += c[q];
        }
    }
    if (g0 + kBkScanItems <= nb_total) {
        *reinterpret_cast<uint4*>(counts + g0) = make_uint4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<uint4*>(counts + g0 + 4) = make_uint4(o[4], o[5], o[6], o[7]);
    } else {
#pragma unroll
        for (int q = 0; q < kBkScanItems; ++q)
            if (g0 + q < nb_total) counts[g0 + q] = o[q];
    }
}

// ordering key of a point inside its bucket: leaf (z cell, column) — or the column alone in a pass-through frame, where
// every point is its own voxel — then the scan position.  (i, j, k) = the point's leaf cell.
__device__ __forceinline__ unsigned long long bk_key64(const BkFrame& B, bool pass, int ci, int cj, int ck, uint32_t ps,
                                                       uint32_t& col) {
    const int bi = ci - B.i0c, bj = cj - B.j0c;
    col = (uint32_t)(bi - (bi / kBkB) * kBkB) + (uint32_t)(bj - (bj / kBkB) * kBkB) * kBkB;
    const uint32_t k32 = pass ? col : (uint32_t)(ck - B.k0) * kBkSub + col;
    return ((unsigned long long)k32 << 32) | ps;
}
__device__ __forceinline__ uint32_t bk_key_col(unsigned long long key, bool pass) {
    const uint32_t k32 = (uint32_t)(key >> 32);
    return pass ? k32 : k32 % (uint32_t)kBkSub;
}

// Shared-memory staging of a warp's 128 samples: a lane writes its (up to) four consecutive records, later lane t reads
// record 32 k + t.  Position p of an array of 16- / 8- / 4-byte records lives at p ^ swizzle(p), which spreads the
// writers' 64- / 32- / 16-byte strides over all banks and keeps the readers' consecutive positions conflict-free.
__device__ __forceinline__ uint32_t swz16(uint32_t p) { return p ^ ((p >> 3) & 3u); }
__device__ __forceinline__ uint32_t swz8(uint32_t p) { return p ^ ((p >> 4) & 3u); }
__device__ __forceinline__ uint32_t swz4(uint32_t p) { return p ^ ((p >> 5) & 3u); }

// ---- pass 2: evaluate again, colour, bin into the buckets ---------------------------------------------------------------
// Every warp works on its 128 consecutive samples alone (no CTA barrier after the table load): compaction by warp prefix,
// staging in the warp's slice of shared memory, one atomic per run of consecutive points of one bucket (issued by the run's
// last point), coalesced copy-out of {x, y, z, rgb} (16 B) + ordering key (8 B: leaf key | scan position).
// The scan position (keypoints, then the row-major grid) is the order PCL's stable grouping (the oracle's) adds the points
// of a leaf in.
constexpr int kBkWarpItems = 128;
struct BkScatterWarp {
    float4 pts[kBkWarpItems];
    unsigned long long key[kBkWarpItems];
    uint32_t bkt[kBkWarpItems];    // bucket of the staged point, then its destination slot
    uint32_t base[kBkWarpItems];   // by run head position: first slot of the run
};
template <int DT>
__global__ void __launch_bounds__(kThreads, 5) k_bk_scatter(AParams P, const FrameDev* __restrict__ frames,
                                                         const BkFrame* __restrict__ bk, const uint8_t* __restrict__ frame_pass,
                                                         float inv_f, uint32_t* __restrict__ cursor, float4* __restrict__ pts,
                                                         unsigned long long* __restrict__ keys_out,
                                                         const uint32_t* __restrict__ flags) {
    wait_prior();
    __shared__ double rl[256];
    __shared__ float zl[256];
    __shared__ __align__(16) BkScatterWarp s_w[kWarps];
    if (*flags) return;   // the histogram already overflowed: the host reruns the batch through the sort engine
    const int tile = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const unsigned lt = (1u << lane) - 1u;
    const FrameDev& F = frames[f];
    const BkFrame B = bk[f];
    const bool pass = frame_pass[f] != 0;
    BkScatterWarp& W = s_w[tid >> 5];
    load_lut(P, rl, zl);
    Samp S;
    eval4<DT>(P, F, rl, zl, tile, S);
    const uint32_t nv = (uint32_t)__popc(S.mask);
    uint32_t inc = nv;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += t;
    }
    const uint32_t total = __shfl_sync(kFull, inc, 31);
    if (total == 0) return;   // (warp-uniform)
    if (S.mask) {
        uint32_t rgb[4];
        if (S.vec_row) {
            const uint32_t* c = reinterpret_cast<const uint32_t*>(F.bgr + (size_t)S.py[0] * F.bgr_step + 3 * (size_t)S.px[0]);
            const uint32_t w0 = __ldcs(c), w1 = __ldcs(c + 1), w2 = __ldcs(c + 2);
            rgb[0] = w0 & 0x00ffffffu;
            rgb[1] = (w0 >> 24) | ((w1 & 0xffffu) << 8);
            rgb[2] = (w1 >> 16) | ((w2 & 0xffu) << 16);
            rgb[3] = w2 >> 8;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (S.mask & (1u << j)) {
                    const uint8_t* c = F.bgr + (size_t)S.py[j] * F.bgr_step + 3 * (size_t)S.px[j];
                    rgb[j] = ((uint32_t)c[2] << 16) | ((uint32_t)c[1] << 8) | (uint32_t)c[0];
                }
        }
        // scan position: keypoint index, or n_kp + grid sample index
        const uint32_t p0 = tile < P.kp_tiles ? (uint32_t)tile * kTileA + tid * 4
                                              : (uint32_t)F.n_kp + (uint32_t)(tile - P.kp_tiles) * kTileA + tid * 4;
        uint32_t o = inc - nv;
        bool bad = false;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (S.mask & (1u << j)) {
                float tx, ty, tz;
                xform(F.T, S.x[j], S.y[j], S.z[j], tx, ty, tz);
                int ci, cj, ck;
                bk_cell(tx, ty, tz, inv_f, ci, cj, ck);
                uint32_t col;
                W.pts[swz16(o)] = make_float4(tx, ty, tz, __uint_as_float(rgb[j]));
                W.key[swz8(o)] = bk_key64(B, pass, ci, cj, ck, p0 + j, col);
                W.bkt[swz4(o)] = bk_index(B, ci, cj, ck, bad);
                ++o;
            }
    }
    __syncwarp();
    // ---- runs of consecutive staged points of one bucket: the run's last point reserves the slots
    const uint32_t e0 = lane * 4;
    uint32_t b[6];   // b[1 + j] = bucket of staged point e0 + j; b[0] / b[5] = the neighbours
#pragma unroll
    for (int j = -1; j <= 4; ++j) {
        const uint32_t e = e0 + j;   // (wraps for e0 == 0, j == -1: e < total is then false)
        b[j + 1] = e < total ? W.bkt[swz4(e)] : 0xffffffffu;
    }
    uint32_t lh = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (e0 + j < total && b[j + 1] != b[j]) lh = e0 + j;
    uint32_t L = lh;   // head of the run that is open when this lane's points begin: exclusive max scan over the lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(kFull, L, o);
        if (lane >= o) L = max(L, t);
    }
    L = __shfl_up_sync(kFull, L, 1);
    if (lane == 0) L = 0;
    uint32_t hp[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t e = e0 + j;
        hp[j] = 0;
        if (e < total) {
            if (b[j + 1] != b[j]) L = e;
            hp[j] = L;
            if (b[j + 2] != b[j + 1]) W.base[L] = atomicAdd(&cursor[b[j + 1]], e - L + 1u);
        }
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t e = e0 + j;
        if (e < total) W.bkt[swz4(e)] = W.base[hp[j]] + (e - hp[j]);
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t t = k * 32 + lane;
        if (t < total) {
            const uint32_t g = W.bkt[swz4(t)];
            pts[g] = W.pts[swz16(t)];
            keys_out[g] = W.key[swz8(t)];
        }
    }
    (void)lt;
}

// ---- pass 3: buckets -> per-frame voxel centroids -> one partial sum per combined-grid cell ------------------------------
// A CTA takes kRdG consecutive non-empty buckets (~1000 points) per ticket and works on all of them at once, one THREAD per
// point in every phase:
//   load      point + ordering key into shared memory; bin = (bucket, leaf column); one shared-memory atomic per point numbers
//             it inside its bin (the arrival order is arbitrary: the rank below orders)
//   scan      first position of every bin
//   rank      each point counts the keys of its bin (3 points on average) that precede its own (leaf key, scan position):
//             final position = PCL's order (column, z cell, scan position) inside the bucket
//   fold      each run head left-folds its leaf in scan order (bit-identical centroid: the oracle's stable order), cells the
//             centroid on the combined grid and leaves it in shared memory
//   sum       one warp per bucket adds the centroids that fell into the bucket's nominal combined cell — lanes in position
//             order, then an xor butterfly: a fixed tree — and writes the partial cell to slot r of the chunk's list
// Centroids that land in a neighbour of the nominal cell (they sit on its border to the last float bit: a couple per frame) are
// "strays": single-centroid records appended behind the main slots through an atomic counter and put into a canonical order
// afterwards (k_bk_strays), so the partial list is reproducible.
constexpr int kRdG = 12;                          // buckets per ticket
constexpr int kRdItems = 5;                       // points per thread
constexpr int kRdCap = kThreads * kRdItems;       // points a CTA holds at once
constexpr int kRdBins = kRdG * kBkSub;
constexpr int kRdStray = 4;                       // strays per bucket kept in shared memory

struct RdSmem {
    float4 pts[kRdCap];                    // load order; a run head's slot is overwritten by its centroid (z + 500)
    unsigned long long skey[kRdCap];       // bin order: (leaf key << 32 | scan position)
    uint32_t fkey[kRdCap];                 // final order: leaf key
    uint16_t sidx[kRdCap];                 // bin order: load index
    uint16_t fidx[kRdCap];                 // final order: load index | 0x8000 head in the nominal cell | 0x4000 stray head
    uint32_t bin[kRdBins + 4];             // per bin: count, then first position ([n_bins] = total)
    uint32_t startbits[kRdCap / 32 + 1];   // bit p: position p starts a bin
    uint4 ent[kRdG];
    uint8_t pass[kRdG];                    // per bucket: its frame passes through PCL's guard (looked up by frame index)
    uint32_t bstart[kRdG + 1];             // first point of each bucket, relative to the sub-batch
    uint8_t cb[kRdCap / 32 + 4];           // bucket that holds position 32 c (the lookup walks on from there)
    uint32_t sub_b1, sub_n;                // the sub-batch: buckets [b0, sub_b1), sub_n points
    int kz[kRdG];                          // z cell of the nominal combined cell
    o3r_cell stray[kRdG][kRdStray];
    uint32_t nstray[kRdG];
    uint32_t scan[34];
    uint32_t ticket;
    int bb[6];
};
constexpr size_t bk_reduce_smem() { return sizeof(RdSmem); }

// x / n for a small positive integer n, bit-identical to IEEE division (what pcl::CentroidPoint's `/ n` compiles to): with
// r = RN(1 / n), q = RN(x r), the residual x - n q is exact in an FMA and one correction step lands on RN(x / n) (Markstein);
// the guard sends anything near the ends of the exponent range, and large n, to the generic division.
__device__ __forceinline__ float bk_div_small(float x, float fn, float r) {
    const float q = __fmul_rn(x, r);
    const float e = __fmaf_rn(-fn, q, x);
    return __fmaf_rn(e, r, q);
}
// pcl::CentroidPoint<PointXYZRGB>: float sums / (float)n; colour uint32(float sum / n) = integer division for these ranges
__device__ __forceinline__ float4 bk_centroid(float sx, float sy, float sz, uint32_t n, uint32_t r, uint32_t g, uint32_t b) {
    const float fn = (float)n;
    float cx, cy, cz;
    uint32_t rgb;
    const float lim_lo = 1e-30f, lim_hi = 1e30f;
    const float ax = fabsf(sx), ay = fabsf(sy), az = fabsf(sz);
    const bool fast = n <= 1024u && (ax == 0.f || (ax > lim_lo && ax < lim_hi)) && (ay == 0.f || (ay > lim_lo && ay < lim_hi)) &&
                      (az == 0.f || (az > lim_lo && az < lim_hi));
    if (fast) {
        const float rc = __frcp_rn(fn);
        cx = bk_div_small(sx, fn, rc); cy = bk_div_small(sy, fn, rc); cz = bk_div_small(sz, fn, rc);
        // channel sums s <= 255 n are integers: uint32((float)s / fn) == floor(s / n), and s * rc + rc / 2 lies within 1e-4 of
        // s / n + 1 / (2 n), whose floor is the same integer (n <= 1024)
        const float h = __fmul_rn(0.5f, rc);
        rgb = ((uint32_t)__fmaf_rn((float)r, rc, h) << 16) | ((uint32_t)__fmaf_rn((float)g, rc, h) << 8) | (uint32_t)__fmaf_rn((float)b, rc, h);
    } else {
        cx = __fdiv_rn(sx, fn); cy = __fdiv_rn(sy, fn); cz = __fdiv_rn(sz, fn);
        rgb = ((uint32_t)__fdiv_rn((float)r, fn) << 16) | ((uint32_t)__fdiv_rn((float)g, fn) << 8) | (uint32_t)__fdiv_rn((float)b, fn);
    }
    return make_float4(cx, cy, cz, __uint_as_float(rgb));
}

__device__ __forceinline__ bool bk_cell_less(const o3r_cell& a, const o3r_cell& b) {
    if (a.key != b.key) return a.key < b.key;
    const uint32_t av[7] = {__float_as_uint(a.sx), __float_as_uint(a.sy), __float_as_uint(a.sz), a.n, a.sr, a.sg, a.sb};
    const uint32_t bv[7] = {__float_as_uint(b.sx), __float_as_uint(b.sy), __float_as_uint(b.sz), b.n, b.sr, b.sg, b.sb};
#pragma unroll
    for (int i = 0; i < 7; ++i)
        if (av[i] != bv[i]) return av[i] < bv[i];
    return false;
}

// out[*out_base + r]            main partial of the r-th non-empty bucket (r < totals[1])
// out[*out_base + totals[1] + ...]  strays, appended through *stray_cnt (at most stray_cap)
__global__ void __launch_bounds__(kThreads, O3R_BK_MINB) k_bk_reduce(
    const float4* __restrict__ pts, const unsigned long long* __restrict__ keys, const uint4* __restrict__ nl,
    const uint8_t* __restrict__ frame_pass, const uint32_t* __restrict__ totals, float icx, float icz, o3r_cell* __restrict__ out,
    const uint32_t* __restrict__ out_base, uint32_t* __restrict__ stray_cnt, uint32_t stray_cap, uint32_t* __restrict__ ticket,
    uint32_t* __restrict__ frame_vox, int* __restrict__ cellbb, uint32_t* __restrict__ flags, float4* __restrict__ dbg_vox,
    uint32_t* __restrict__ dbg_cnt) {
    wait_prior();
    extern __shared__ __align__(16) unsigned char bk_smem_raw[];
    RdSmem& S = *reinterpret_cast<RdSmem*>(bk_smem_raw);
    if (flags[0]) return;   // raised by the histogram / scan (complete before this kernel starts): uniform exit
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t NR = totals[1];
    o3r_cell* const out0 = out + *out_base;
    if (tid < 6) S.bb[tid] = tid < 3 ? 0x7fffffff : (int)0x80000000;
    // range of combined-grid cells touched (the merge packs its sort keys into it)
    int cmn[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff}, cmx[3] = {(int)0x80000000, (int)0x80000000, (int)0x80000000};
    const int Bi = 1 << 20;
    for (;;) {
        __syncthreads();   // (the previous ticket's shared memory is free)
        if (tid == 0) S.ticket = atomicAdd(ticket, (uint32_t)kRdG);
        __syncthreads();
        const uint32_t r0 = S.ticket;
        if (r0 >= NR) break;
        const int nb = (int)min((uint32_t)kRdG, NR - r0);
        if (tid < nb) {
            const uint4 e = nl[r0 + tid];
            S.ent[tid] = e;
            S.pass[tid] = frame_pass[e.y >> 16];
        }
        __syncthreads();
        for (int b0 = 0; b0 < nb;) {
            // ---- sub-batch: as many of the ticket's buckets as fit (normally all of them)
            const uint32_t base = S.ent[b0].x;
            __syncthreads();   // (the previous sub-batch is done with shared memory)
            if (tid == 0) {
                int e1 = b0;
                uint32_t m = 0;
                while (e1 < nb) {
                    const uint32_t c = S.ent[e1].y & 0xffffu;
                    if (m + c > (uint32_t)kRdCap) break;
                    m += c; ++e1;
                }
                S.sub_b1 = (uint32_t)e1; S.sub_n = m;
            }
            __syncthreads();
            const int b1 = (int)S.sub_b1;
            const uint32_t n = S.sub_n;
            if (b1 == b0) {   // a single bucket larger than a CTA can hold: give up (the host falls back to the sort engine)
                if (tid == 0) atomicOr(flags + 1, BK_FLAG_BUCKET);
                ++b0;
                continue;
            }
            const int nbb = b1 - b0, nbins = nbb * kBkSub;
            for (int i = tid; i <= nbins; i += kThreads) S.bin[i] = 0u;
            for (int i = tid; i < kRdCap / 32 + 1; i += kThreads) S.startbits[i] = 0u;
            if (tid <= nbb) S.bstart[tid] = tid < nbb ? S.ent[b0 + tid].x - base : n;
            if (tid < nbb) S.nstray[tid] = 0u;
            __syncthreads();
            if (tid * 32u < n + 32u) {   // coarse position -> bucket table
                const uint32_t i = tid * 32u;
                int bl = 0;
#pragma unroll
                for (int st = 8; st > 0; st >>= 1)
                    if (bl + st < nbb && S.bstart[bl + st] <= i) bl += st;
                S.cb[tid] = (uint8_t)bl;
            }
            __syncthreads();
            // ---- load; number every point inside its (bucket, column) bin
            unsigned long long key[kRdItems];
            uint32_t bs[kRdItems];   // bin | slot << 16
#pragma unroll
            for (int k = 0; k < kRdItems; ++k) {
                const uint32_t i = k * kThreads + tid;
                if (i < n) {
                    key[k] = __ldcs(keys + base + i);
                    S.pts[i] = __ldcs(pts + base + i);
                    int bl = S.cb[i >> 5];
                    while (bl + 1 < nbb && S.bstart[bl + 1] <= i) ++bl;
                    const bool pass = S.pass[b0 + bl] != 0;
                    const uint32_t bin = (uint32_t)bl * kBkSub + bk_key_col(key[k], pass);
                    bs[k] = bin | (atomicAdd(&S.bin[bin], 1u) << 16);
                }
            }
            __syncthreads();
            {   // first position of every bin; mark where bins start
                const int i0 = tid * 2;
                const uint32_t c0 = i0 < nbins ? S.bin[i0] : 0u, c1 = i0 + 1 < nbins ? S.bin[i0 + 1] : 0u;
                uint32_t tot;
                const uint32_t ex = block_excl_scan(c0 + c1, S.scan, tot);
                if (i0 < nbins) { S.bin[i0] = ex; if (c0) atomicOr(&S.startbits[ex >> 5], 1u << (ex & 31u)); }
                if (i0 + 1 < nbins) { S.bin[i0 + 1] = ex + c0; if (c1) atomicOr(&S.startbits[(ex + c0) >> 5], 1u << ((ex + c0) & 31u)); }
                if (tid == 0) S.bin[nbins] = n;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < kRdItems; ++k) {
                const uint32_t i = k * kThreads + tid;
                if (i < n) {
                    const uint32_t at = S.bin[bs[k] & 0xffffu] + (bs[k] >> 16);
                    S.skey[at] = key[k];
                    S.sidx[at] = (uint16_t)i;
                }
            }
            __syncthreads();
            // ---- rank inside the bin by (leaf key, scan position)
#pragma unroll
            for (int k = 0; k < kRdItems; ++k) {
                const uint32_t i = k * kThreads + tid;
                if (i < n) {
                    const uint32_t bin = bs[k] & 0xffffu;
                    const uint32_t a = S.bin[bin], e = S.bin[bin + 1];
                    uint32_t rk = a;
#pragma unroll 2
                    for (uint32_t j = a; j < e; ++j) rk += S.skey[j] < key[k] ? 1u : 0u;
                    S.fkey[rk] = (uint32_t)(key[k] >> 32);
                    S.fidx[rk] = (uint16_t)i;
                }
            }
            __syncthreads();
            // z cell of each bucket's nominal combined cell: that of its first point in final order
            if (tid < nbb) {
                const float4 p = S.pts[S.fidx[S.bstart[tid]]];
                S.kz[tid] = (int)floorf(__fmul_rn(__fadd_rn(p.z, 500.0f), icz));
            }
            __syncthreads();
            // ---- leaves: left fold in scan order; combined-grid cell of every centroid
#pragma unroll 1
            for (int k = 0; k < kRdItems; ++k) {
                const uint32_t pos = k * kThreads + tid;
                if (pos >= n) break;
                int bl = S.cb[pos >> 5];
                while (bl + 1 < nbb && S.bstart[bl + 1] <= pos) ++bl;
                const uint4 ent = S.ent[b0 + bl];
                const bool pass = S.pass[b0 + bl] != 0;
                const uint32_t k32 = S.fkey[pos];
                const bool head = pass || ((S.startbits[pos >> 5] >> (pos & 31u)) & 1u) || S.fkey[pos - 1] != k32;
                if (!head) continue;
                const uint32_t me = S.fidx[pos];
                float4 p = S.pts[me];
                float4 cen;
                if (pass) {
                    cen = p;   // PCL: output = *input_
                } else {
                    float sx = 0.f, sy = 0.f, sz = 0.f;
                    uint32_t cn = 0, cr = 0, cg = 0, cb = 0;
                    uint32_t q = pos;
                    for (;;) {
                        sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z);
                        const uint32_t w = __float_as_uint(p.w);
                        cr += (w >> 16) & 255u; cg += (w >> 8) & 255u; cb += w & 255u;
                        ++cn; ++q;
                        if (q >= n || ((S.startbits[q >> 5] >> (q & 31u)) & 1u) || S.fkey[q] != k32) break;
                        p = S.pts[S.fidx[q]];
                    }
                    cen = bk_centroid(sx, sy, sz, cn, cr, cg, cb);
                }
                if (dbg_vox) dbg_vox[atomicAdd(dbg_cnt, 1u)] = cen;
                cen.z = __fadd_rn(cen.z, 500.0f);   // pose_functions.cpp:1666
                const int vi = (int)floorf(__fmul_rn(cen.x, icx)), vj = (int)floorf(__fmul_rn(cen.y, icx)),
                          vk = (int)floorf(__fmul_rn(cen.z, icz));
                if (vi == (int)ent.z && vj == (int)ent.w && vk == S.kz[bl]) {
                    S.pts[me] = cen;
                    S.fidx[pos] = (uint16_t)(me | 0x8000u);
                } else {   // on the border of the nominal cell to the last float bit: its own record
                    S.fidx[pos] = (uint16_t)(me | 0x4000u);
                    cmn[0] = min(cmn[0], vi); cmx[0] = max(cmx[0], vi);
                    cmn[1] = min(cmn[1], vj); cmx[1] = max(cmx[1], vj);
                    cmn[2] = min(cmn[2], vk); cmx[2] = max(cmx[2], vk);
                    const uint32_t sl = atomicAdd(&S.nstray[bl], 1u);
                    if (sl < (uint32_t)kRdStray) {
                        const uint32_t w = __float_as_uint(cen.w);
                        o3r_cell pc;
                        pc.key = ((unsigned long long)(uint32_t)(vk + Bi) << 42) | ((unsigned long long)(uint32_t)(vj + Bi) << 21) |
                                 (unsigned long long)(uint32_t)(vi + Bi);
                        pc.sx = cen.x; pc.sy = cen.y; pc.sz = cen.z; pc.n = 1u;
                        pc.sr = (w >> 16) & 255u; pc.sg = (w >> 8) & 255u; pc.sb = w & 255u; pc.pad = 0u;
                        S.stray[bl][sl] = pc;
                    }
                }
            }
            __syncthreads();
            // ---- one warp per bucket: the partial sum of the nominal cell (lanes in position order, then an xor butterfly)
            for (int bl = warp; bl < nbb; bl += kWarps) {
                const uint4 ent = S.ent[b0 + bl];
                const uint32_t a = S.bstart[bl], e = S.bstart[bl + 1];
                float ax = 0.f, ay = 0.f, az = 0.f;
                uint32_t an = 0, ar = 0, ag = 0, ab = 0, nh = 0;
                for (uint32_t pos = a + lane; pos < e; pos += 32) {
                    const uint32_t fi = S.fidx[pos];
                    if (fi & 0x8000u) {
                        const float4 c = S.pts[fi & 0x3fffu];
                        const uint32_t w = __float_as_uint(c.w);
                        ax = __fadd_rn(ax, c.x); ay = __fadd_rn(ay, c.y); az = __fadd_rn(az, c.z);
                        ++an; ar += (w >> 16) & 255u; ag += (w >> 8) & 255u; ab += w & 255u;
                    }
                    nh += (fi & 0xc000u) ? 1u : 0u;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    ax = __fadd_rn(ax, __shfl_xor_sync(kFull, ax, o));
                    ay = __fadd_rn(ay, __shfl_xor_sync(kFull, ay, o));
                    az = __fadd_rn(az, __shfl_xor_sync(kFull, az, o));
                }
                an = __reduce_add_sync(kFull, an); ar = __reduce_add_sync(kFull, ar);
                ag = __reduce_add_sync(kFull, ag); ab = __reduce_add_sync(kFull, ab);
                nh = __reduce_add_sync(kFull, nh);
                if (lane == 0) {
                    uint32_t ns = S.nstray[bl];
                    if (ns > (uint32_t)kRdStray) { atomicOr(flags + 1, BK_FLAG_PART); ns = kRdStray; }
                    o3r_cell mainc;
                    const int nI = (int)ent.z, nJ = (int)ent.w, kz = S.kz[bl];
                    mainc.key = ((unsigned long long)(uint32_t)(kz + Bi) << 42) | ((unsigned long long)(uint32_t)(nJ + Bi) << 21) |
                                (unsigned long long)(uint32_t)(nI + Bi);
                    mainc.sx = ax; mainc.sy = ay; mainc.sz = az; mainc.n = an; mainc.sr = ar; mainc.sg = ag; mainc.sb = ab; mainc.pad = 0u;
                    if (an == 0u) {   // every centroid strayed: no empty record — the smallest stray takes the main slot
                        uint32_t best = 0;
                        for (uint32_t i = 1; i < ns; ++i)
                            if (bk_cell_less(S.stray[bl][i], S.stray[bl][best])) best = i;
                        mainc = S.stray[bl][best];
                        S.stray[bl][best] = S.stray[bl][ns - 1];
                        --ns;
                    } else {
                        cmn[0] = min(cmn[0], nI); cmx[0] = max(cmx[0], nI);
                        cmn[1] = min(cmn[1], nJ); cmx[1] = max(cmx[1], nJ);
                        cmn[2] = min(cmn[2], kz); cmx[2] = max(cmx[2], kz);
                    }
                    out0[r0 + b0 + bl] = mainc;
                    atomicAdd(&frame_vox[ent.y >> 16], nh);
                    if (ns) {
                        const uint32_t at = atomicAdd(stray_cnt, ns);
                        if (at + ns > stray_cap) atomicOr(flags + 1, BK_FLAG_PART);
                        else
                            for (uint32_t i = 0; i < ns; ++i) out0[NR + at + i] = S.stray[bl][i];
                    }
                }
            }
            b0 = b1;
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int lo = __reduce_min_sync(kFull, cmn[a]), hi = __reduce_max_sync(kFull, cmx[a]);
        cmn[a] = lo; cmx[a] = hi;
    }
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { atomicMin(&S.bb[a], cmn[a]); atomicMax(&S.bb[3 + a], cmx[a]); }
    }
    __syncthreads();
    if (tid < 3) { if (S.bb[tid] != 0x7fffffff) atomicMin(&cellbb[tid], S.bb[tid]); }
    else if (tid < 6) { if (S.bb[tid] != (int)0x80000000) atomicMax(&cellbb[tid], S.bb[tid]); }
}

// Canonical order of the chunk's stray records (they were appended in atomic order): rank by the whole record.  Two records
// that compare equal are identical, so their mutual order does not matter.  One CTA; n is tiny (a couple per frame).
// Also publishes the chunk's record count: main slots + strays.
__global__ void __launch_bounds__(1024) k_bk_strays(o3r_cell* __restrict__ out, const uint32_t* __restrict__ out_base,
                                                    const uint32_t* __restrict__ totals, const uint32_t* __restrict__ stray_cnt,
                                                    uint32_t stray_cap, o3r_cell* __restrict__ tmp, uint32_t* __restrict__ chunk_total,
                                                    const uint32_t* __restrict__ flags) {
    wait_prior();
    if (flags[0]) { if (threadIdx.x == 0) *chunk_total = 0u; return; }
    const uint32_t NR = totals[1], n = min(*stray_cnt, stray_cap);
    if (threadIdx.x == 0) *chunk_total = NR + n;
    if (n < 2) return;
    o3r_cell* s = out + *out_base + NR;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        const o3r_cell me = s[i];
        uint32_t rk = 0;
        for (uint32_t j = 0; j < n; ++j) {
            const o3r_cell o = s[j];
            rk += (bk_cell_less(o, me) || (!bk_cell_less(me, o) && j < i)) ? 1u : 0u;
        }
        tmp[rk] = me;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s[i] = tmp[i];
}

}  // namespace o3r
