// sor.cuh — pcl::StatisticalOutlierRemoval (pose_functions.cpp:1673-1686: setMeanK(50), setStddevMulThresh(1.0)), the
// filter the reference applies to every frame's cloud before the per-frame VoxelGrid whenever jump_pixels > 0.
//
// PCL: for every point the mean_k + 1 nearest neighbours by exact k-NN (KdTreeFLANN, flann::L2_Simple<float>:
// d2 = ((dx*dx) + (dy*dy)) + (dz*dz) in float), dist_i = (float)(sum_{k=1..mean_k} sqrt((double)d2_k) / mean_k) with the
// neighbours in ascending order (k = 0 is the query), then mean and stddev of dist over the cloud in double and
// "remove iff dist_i > mean + mul * stddev".  An exact k-NN does not depend on how it is found; here:
//   * a uniform grid per frame, points radix-sorted by cell index (x minor) and a start offset per CELL (the classic
//     uniform-grid layout): "all points in cells [a, b] of a (y, z) row" is one contiguous range found with two
//     independent loads — no per-row search, no key compares in the candidate loop (a per-row table with a binary
//     search was the first version: each of the ~30 rows a query visits cost a chain of 6-8 dependent loads, which
//     is what bounded the kernel);
//   * one thread per query, in cell order (a warp's queries share their candidate rows): the cube of (2s+1)^3 cells
//     around the query is scanned into a per-thread max-heap of the mean_k + 1 smallest d2 (shared memory), s grows until
//     the heap's top provably lies inside the cube (every unscanned point is farther than (s - 0.05) cells);
//   * heapsort in place, sum in ascending order -> the same double additions as the CPU loop, bit for bit.
// The cloud statistics are reduced in a fixed tree order (the reference adds sequentially: ~1e-13 relative on the
// threshold, which only matters for a point whose distance equals the threshold to 13 digits).
#pragma once
#include "common.cuh"
#include "sort.cuh"

namespace o3r {

constexpr int kSorThreads = 128;
constexpr int kSorCellsCap = 1 << 22;  // cells per frame (4 M start offsets = 16 MB); the cell is enlarged until they fit
constexpr int kSorMaxK = 128;          // mean_k + 1 <= 128
#ifndef O3R_SOR_CALIB_RANK
#define O3R_SOR_CALIB_RANK 115
#endif
constexpr int kSorCalibRank = O3R_SOR_CALIB_RANK;   // which of the 128 sorted sample radii sizes the cell (115 = 90th percentile; measured: the median makes the hard phase 3x longer)

struct SorGrid {
    float mn[3];
    float inv, c;
    int nc[3];
    int empty;
};

// per frame: cell size and table shape from the frame's bbox ({minx,miny,minz,maxx,maxy,maxz} as ordered uints) and count.
// Also fills the GridParams fields the radix-sort planner reads (key_bits, passthrough, empty).
__global__ void k_sor_grid(int n_seg, const uint32_t* __restrict__ bbox, const uint32_t* __restrict__ seg_off, int mean_k,
                           SorGrid* __restrict__ grids, GridParams* __restrict__ plan_grids) {
    wait_prior();
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const uint32_t n = seg_off[s + 1] - seg_off[s];
    SorGrid G;
    GridParams P;
    memset(&P, 0, sizeof(P));
    G.empty = (n == 0) || bbox[6 * s] == 0xffffffffu;
    G.inv = 1.f; G.c = 1.f;
    G.nc[0] = G.nc[1] = G.nc[2] = 1;
    G.mn[0] = G.mn[1] = G.mn[2] = 0.f;
    P.empty = G.empty;
    P.key_bits = 1;
    if (!G.empty) {
        double ext[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            G.mn[a] = ord2f(bbox[6 * s + a]);
            ext[a] = (double)ord2f(bbox[6 * s + 3 + a]) - (double)G.mn[a];
        }
        const double e_hi = fmax(ext[0], fmax(ext[1], ext[2])), e_lo = fmin(ext[0], fmin(ext[1], ext[2]));
        const double e_mid = ext[0] + ext[1] + ext[2] - e_hi - e_lo;
        const double area = fmax(e_hi * e_mid, 1e-12);
        double c = sqrt((double)(mean_k + 1) * area / (3.141592653589793 * (double)n));
        c = fmax(c, 1e-6);
        long long nc[3];
        for (;;) {
#pragma unroll
            for (int a = 0; a < 3; ++a) nc[a] = (long long)(ext[a] / c) + 2;
            if (nc[0] * nc[1] * nc[2] <= (long long)kSorCellsCap) break;
            c *= 1.26;
        }
        G.c = (float)c;
        G.inv = (float)(1.0 / c);
        G.nc[0] = (int)nc[0]; G.nc[1] = (int)nc[1]; G.nc[2] = (int)nc[2];
        const long long cells = nc[0] * nc[1] * nc[2];
        P.key_bits = cells > 1 ? 64 - __clzll(cells - 1) : 1;
    }
    grids[s] = G;
    plan_grids[s] = P;
}

__device__ __forceinline__ uint32_t sor_cell(const SorGrid& G, float x, float y, float z) {
    const int ix = min(G.nc[0] - 1, max(0, (int)floorf(__fmul_rn(__fsub_rn(x, G.mn[0]), G.inv))));
    const int iy = min(G.nc[1] - 1, max(0, (int)floorf(__fmul_rn(__fsub_rn(y, G.mn[1]), G.inv))));
    const int iz = min(G.nc[2] - 1, max(0, (int)floorf(__fmul_rn(__fsub_rn(z, G.mn[2]), G.inv))));
    return (uint32_t)ix + (uint32_t)G.nc[0] * ((uint32_t)iy + (uint32_t)G.nc[1] * (uint32_t)iz);
}

__global__ void __launch_bounds__(kThreads) k_sor_key(const float4* __restrict__ pts, const uint32_t* __restrict__ seg_off,
                                                      const SorGrid* __restrict__ grids, uint32_t* __restrict__ keys) {
    wait_prior();
    const int s = blockIdx.y;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    const SorGrid G = grids[s];
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        const float4 p = pts[beg + i];
        keys[beg + i] = sor_cell(G, p.x, p.y, p.z);
    }
}

// sorted keys -> start offset of every cell (cell_start[c] = first sorted position whose key is >= c, cell_start[cells] = n;
// positions relative to the segment); also copies the sorted keys, values and points out of the sort's ping-pong
// buffers (which side holds a segment's result is per segment).  Position i owns the cells (key[i-1], key[i]]; most cells of
// a surface's bounding box are empty, so those gaps are long (whole rows of cells): gaps of more than 4 cells are filled by
// the whole warp with coalesced stores, and the cells behind the last key by the whole grid.
__global__ void __launch_bounds__(kThreads) k_sor_cells(const uint32_t* __restrict__ keys0, const uint32_t* __restrict__ keys1,
                                                        const uint32_t* __restrict__ vals0, const uint32_t* __restrict__ vals1,
                                                        const SortPlan* __restrict__ plan, const float4* __restrict__ pts,
                                                        const uint32_t* __restrict__ seg_off, const SorGrid* __restrict__ grids,
                                                        uint32_t* __restrict__ cell_start, uint32_t* __restrict__ skeys,
                                                        uint32_t* __restrict__ svals, float4* __restrict__ spts) {
    wait_prior();
    const int s = blockIdx.y;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    const uint32_t cells = (uint32_t)grids[s].nc[0] * (uint32_t)grids[s].nc[1] * (uint32_t)grids[s].nc[2];
    uint32_t* cs = cell_start + (size_t)s * (kSorCellsCap + 1);
    const int par = plan[s].final_parity;
    const bool ident = plan[s].n_active == 0;   // nothing was sorted: values were never written (identity)
    const uint32_t* keys = (par ? keys1 : keys0) + beg;
    const uint32_t* vals = (par ? vals1 : vals0) + beg;
    const uint32_t gtid = blockIdx.x * kThreads + threadIdx.x, gstride = gridDim.x * kThreads;
    const uint32_t tail = n ? keys[n - 1] + 1u : 0u;
    for (uint32_t c = tail + gtid; c <= cells; c += gstride) cs[c] = n;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t base = gtid - lane; base < n; base += gstride) {   // warp-uniform trip count
        const uint32_t i = base + lane;
        uint32_t first = 0u, len = 0u;
        if (i < n) {
            const uint32_t k = keys[i];
            first = i == 0 ? 0u : keys[i - 1] + 1u;
            len = k + 1u - first;                                    // 0 when key[i] == key[i-1]
            if (len <= 4u)
                for (uint32_t c = 0; c < len; ++c) cs[first + c] = i;
            const uint32_t v = ident ? beg + i : vals[i];
            skeys[beg + i] = k;
            svals[beg + i] = v;
            spts[beg + i] = pts[v];
        }
        uint32_t m = __ballot_sync(kFull, len > 4u);
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1u;
            const uint32_t f = __shfl_sync(kFull, first, src), l = __shfl_sync(kFull, len, src);
            for (uint32_t c = lane; c < l; c += 32u) cs[f + c] = base + (uint32_t)src;
        }
    }
}

#define SOR_H(k) h[(k) * kSorThreads]
// The heap is 4-ary (children of c: 4c+1 .. 4c+4): 3 levels for 51 entries instead of 6, and the four child loads of a
// level are independent, so a sift costs half the dependent shared-memory round trips of a binary heap.
// Sinks value v from position c in a heap of m entries.
__device__ __forceinline__ void sor_sift_down(float* __restrict__ h, int c, const int m, const float v) {
    for (;;) {
        const int ch0 = 4 * c + 1;
        if (ch0 >= m) break;
        float cv = SOR_H(ch0);
        int ch = ch0;
#pragma unroll
        for (int u = 1; u < 4; ++u) {
            if (ch0 + u < m) {
                const float w = SOR_H(ch0 + u);
                if (w > cv) { cv = w; ch = ch0 + u; }
            }
        }
        if (cv <= v) break;
        SOR_H(c) = cv;
        c = ch;
    }
    SOR_H(c) = v;
}
// One pass of the exact (mean_k + 1)-NN search of a query: scans the cube of (2*sh+1)^3 cells around it into the thread's
// max-heap (element k at h[k * kSorThreads]).  Returns true when the result is proven: the heap holds K entries and its
// top lies inside the cube (every unscanned point is farther than (sh - 0.05) cells), or the cube covers the whole grid.
// cnt = heap entries, top = the heap's largest entry when cnt == K.
__device__ __forceinline__ bool sor_pass(const SorGrid& G, const float4 q, const int ix, const int iy, const int iz,
                                         const float4* __restrict__ pseg, const uint32_t* __restrict__ cs, const int K,
                                         float* __restrict__ h, const int sh, int& cnt, float& top) {
    const int nx = G.nc[0], ny = G.nc[1], nz = G.nc[2];
    cnt = 0;
    top = 0.f;
    // rows are visited ring by ring around the query's own row, so the heap's top is close to final after the first
    // few rows and later candidates rarely replace anything; once the heap is full, a row whose (y, z) interval is
    // farther from the query than sqrt(top) is skipped without touching memory (2 % of a cell of slack for the float
    // rounding of the cell assignment)
    const float slack = __fmul_rn(0.02f, G.c);
    for (int ring = 0; ring <= sh; ++ring)
    for (int dz = -ring; dz <= ring; ++dz) {
        const int z = iz + dz;
        if (z < 0 || z >= nz) continue;
        const float zlo = __fadd_rn(G.mn[2], __fmul_rn((float)z, G.c));
        const float gz = fmaxf(0.f, __fsub_rn(fmaxf(__fsub_rn(zlo, q.z), __fsub_rn(q.z, __fadd_rn(zlo, G.c))), slack));
        for (int dy = -ring; dy <= ring; ++dy) {
            if (max(abs(dy), abs(dz)) != ring) continue;
            const int y = iy + dy;
            if (y < 0 || y >= ny) continue;
            int xlo = max(0, ix - sh), xhi = min(nx - 1, ix + sh);
            if (cnt == K) {
                const float ylo = __fadd_rn(G.mn[1], __fmul_rn((float)y, G.c));
                const float gy = fmaxf(0.f, __fsub_rn(fmaxf(__fsub_rn(ylo, q.y), __fsub_rn(q.y, __fadd_rn(ylo, G.c))), slack));
                const float rem = __fsub_rn(top, __fadd_rn(__fmul_rn(gy, gy), __fmul_rn(gz, gz)));
                if (rem < 0.f) continue;
                // only the cells of the row within sqrt(rem) of the query in x can still hold a closer point
                const float dxm = __fadd_rn(sqrtf(rem), slack);
                xlo = max(xlo, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(q.x, dxm), G.mn[0]), G.inv)) - 0);
                xhi = min(xhi, (int)floorf(__fmul_rn(__fsub_rn(__fadd_rn(q.x, dxm), G.mn[0]), G.inv)));
                if (xlo > xhi) continue;
            }
            const uint32_t c0 = (uint32_t)nx * ((uint32_t)y + (uint32_t)ny * (uint32_t)z);
            const uint32_t lo = cs[c0 + (uint32_t)xlo], e = cs[c0 + (uint32_t)xhi + 1u];
            for (uint32_t t = lo; t < e; ++t) {
                const float4 p = pseg[t];
                const float dx = __fsub_rn(q.x, p.x), dy = __fsub_rn(q.y, p.y), dz = __fsub_rn(q.z, p.z);
                const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
                if (cnt < K) {   // sift up
                    int c = cnt++;
                    while (c > 0) {
                        const int par = (c - 1) >> 2;
                        const float pv = SOR_H(par);
                        if (pv >= d2) break;
                        SOR_H(c) = pv;
                        c = par;
                    }
                    SOR_H(c) = d2;
                    if (cnt == K) top = SOR_H(0);
                } else if (d2 < top) {   // replace the largest, sift down
                    sor_sift_down(h, 0, K, d2);
                    top = SOR_H(0);
                }
            }
        }
    }
    const bool all = ix - sh <= 0 && ix + sh >= nx - 1 && iy - sh <= 0 && iy + sh >= ny - 1 && iz - sh <= 0 && iz + sh >= nz - 1;
    const float reach = __fmul_rn((float)sh - 0.05f, G.c);
    return all || (cnt == K && top <= __fmul_rn(reach, reach));
}

// the cube that is certain to prove the result after a pass that did not: the ball of radius sqrt(top) holds K points, so
// the K-th neighbour is no farther; without a full heap the cube just doubles
__device__ __forceinline__ int sor_next_sh(const SorGrid& G, int sh, int cnt, int K, float top) {
    if (cnt == K) return max(sh + 1, (int)ceilf(__fadd_rn(__fmul_rn(sqrtf(top), G.inv), 0.06f)));
    return sh * 2;
}

// full search: passes until proven
__device__ __forceinline__ int sor_query(const SorGrid& G, const float4 q, const int ix, const int iy, const int iz,
                                         const float4* __restrict__ pseg, const uint32_t* __restrict__ cs, const int K,
                                         float* __restrict__ h, int sh, float& top) {
    int cnt;
    while (!sor_pass(G, q, ix, iy, iz, pseg, cs, K, h, sh, cnt, top)) sh = sor_next_sh(G, sh, cnt, K, top);
    return cnt;
}

// heapsort in place (ascending; element 0 is the query itself, 0.0), then PCL's sum over k = 1 .. in that order
__device__ __forceinline__ float sor_mean_distance(float* __restrict__ h, int cnt, int mean_k) {
    for (int m = cnt - 1; m > 0; --m) {
        const float last = SOR_H(m);
        SOR_H(m) = SOR_H(0);
        sor_sift_down(h, 0, m, last);
    }
    double sum = 0.0;
    for (int k = 1; k < cnt; ++k) sum = __dadd_rn(sum, __dsqrt_rn((double)SOR_H(k)));
    return __double2float_rn(__ddiv_rn(sum, (double)mean_k));
}
#undef SOR_H

// Calibration: the exact (mean_k + 1)-NN radius of 128 evenly spaced sample queries per frame on the first grid (whose
// cell comes from a surface-density guess), and from their 90th percentile the cell of the grid the full search runs on:
// cell = r90 / 1.9, so that the first cube (2 cells each way) already proves the result for ~90 % of the queries while
// holding ~2x the points of the exact ball.  Layered / noisy clouds are several times sparser than the guess assumes.
__global__ void __launch_bounds__(kSorThreads) k_sor_calib(const float4* __restrict__ spts, const uint32_t* __restrict__ keys,
                                                           const uint32_t* __restrict__ seg_off, SorGrid* __restrict__ grids,
                                                           GridParams* __restrict__ plan_grids, const uint32_t* __restrict__ bbox,
                                                           const uint32_t* __restrict__ cell_start, int mean_k) {
    wait_prior();
    extern __shared__ float sor_heap[];
    __shared__ float s_r[kSorThreads];
    __shared__ float s_r90;
    const int s = blockIdx.x;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    const int K = mean_k + 1;
    if (n <= (uint32_t)K) return;   // every query scans the whole cloud anyway
    const SorGrid G = grids[s];
    const uint32_t j = (uint32_t)(((unsigned long long)threadIdx.x * n) / kSorThreads);
    const float4 q = spts[beg + j];
    const uint32_t key = keys[beg + j];
    const int ix = (int)(key % (uint32_t)G.nc[0]), rr = (int)(key / (uint32_t)G.nc[0]), iy = rr % G.nc[1], iz = rr / G.nc[1];
    float* h = sor_heap + threadIdx.x;
    // at most two passes per sample (the second over at most 13^3 cells): a sample that is still unproven is an outlier
    // of the radius distribution and simply ranks last
    float top;
    int cnt;
    const uint32_t* cs = cell_start + (size_t)s * (kSorCellsCap + 1);
    bool ok = sor_pass(G, q, ix, iy, iz, spts + beg, cs, K, h, 2, cnt, top);
    if (!ok) ok = sor_pass(G, q, ix, iy, iz, spts + beg, cs, K, h, min(sor_next_sh(G, 2, cnt, K, top), 6), cnt, top);
    s_r[threadIdx.x] = (ok && cnt == K) ? sqrtf(top) : 3.0e38f;
    if (threadIdx.x == 0) s_r90 = 0.f;
    __syncthreads();
    const float mine = s_r[threadIdx.x];
    int rank = 0;
    for (int t = 0; t < kSorThreads; ++t) rank += (s_r[t] < mine) || (s_r[t] == mine && t < (int)threadIdx.x);
    if (rank == kSorCalibRank) s_r90 = mine;
    __syncthreads();
    if (threadIdx.x == 0 && s_r90 > 0.f && s_r90 < 1.0e38f) {
        double ext[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) ext[a] = (double)ord2f(bbox[6 * s + 3 + a]) - (double)G.mn[a];
        double c = fmax((double)s_r90 / 1.9, 1e-6);
        long long nc[3];
        for (;;) {
#pragma unroll
            for (int a = 0; a < 3; ++a) nc[a] = (long long)(ext[a] / c) + 2;
            if (nc[0] * nc[1] * nc[2] <= (long long)kSorCellsCap) break;
            c *= 1.26;
        }
        SorGrid N = G;
        N.c = (float)c;
        N.inv = (float)(1.0 / c);
        N.nc[0] = (int)nc[0]; N.nc[1] = (int)nc[1]; N.nc[2] = (int)nc[2];
        grids[s] = N;
        const long long cells = nc[0] * nc[1] * nc[2];
        plan_grids[s].key_bits = cells > 1 ? 64 - __clzll(cells - 1) : 1;
    }
}

// Phase 1: one thread per query (sorted position), ONE pass over the 5^3 cube.  Proven queries (~90 %) are finished; the
// others go to the hard list {position in the batch, frame << 16 | cube to scan next}, so that their long searches run in
// warps of their own (phase 2) instead of stalling the 31 easy queries of their warp.
// Dynamic shared memory of both kernels: (mean_k + 1) * kSorThreads floats.
__global__ void __launch_bounds__(kSorThreads) k_sor_knn(const float4* __restrict__ spts, const uint32_t* __restrict__ keys,
                                                         const uint32_t* __restrict__ vals, const uint32_t* __restrict__ seg_off,
                                                         const SorGrid* __restrict__ grids, const uint32_t* __restrict__ cell_start, int mean_k,
                                                         float* __restrict__ dist, uint2* __restrict__ hard,
                                                         uint32_t* __restrict__ n_hard) {
    wait_prior();
    extern __shared__ float sor_heap[];
    const int s = blockIdx.y;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    const uint32_t j = blockIdx.x * kSorThreads + threadIdx.x;
    if (j >= n) return;
    const SorGrid G = grids[s];
    const int K = mean_k + 1;
    float* h = sor_heap + threadIdx.x;
    const float4 q = spts[beg + j];
    const uint32_t key = keys[beg + j];
    const int ix = (int)(key % (uint32_t)G.nc[0]), rr = (int)(key / (uint32_t)G.nc[0]), iy = rr % G.nc[1], iz = rr / G.nc[1];
    int cnt;
    float top;
    if (sor_pass(G, q, ix, iy, iz, spts + beg, cell_start + (size_t)s * (kSorCellsCap + 1), K, h, 2, cnt, top)) {
        dist[vals[beg + j]] = sor_mean_distance(h, cnt, mean_k);
    } else {
        const int sh = min(sor_next_sh(G, 2, cnt, K, top), 65535);
        hard[atomicAdd(n_hard, 1u)] = make_uint2(beg + j, ((uint32_t)s << 16) | (uint32_t)sh);
    }
}

// Phase 2: the hard queries, densely packed.  (Launched over an upper bound; the count is read from the device.)
__global__ void __launch_bounds__(kSorThreads) k_sor_knn_hard(const float4* __restrict__ spts, const uint32_t* __restrict__ keys,
                                                              const uint32_t* __restrict__ vals, const uint32_t* __restrict__ seg_off,
                                                              const SorGrid* __restrict__ grids,
                                                              const uint32_t* __restrict__ cell_start, int mean_k,
                                                              float* __restrict__ dist, const uint2* __restrict__ hard,
                                                              const uint32_t* __restrict__ n_hard) {
    wait_prior();
    extern __shared__ float sor_heap[];
    const uint32_t i = blockIdx.x * kSorThreads + threadIdx.x;
    if (i >= *n_hard) return;
    const uint2 hq = hard[i];
    const int s = (int)(hq.y >> 16);
    const uint32_t beg = seg_off[s];
    const SorGrid G = grids[s];
    const int K = mean_k + 1;
    float* h = sor_heap + threadIdx.x;
    const float4 q = spts[hq.x];
    const uint32_t key = keys[hq.x];
    const int ix = (int)(key % (uint32_t)G.nc[0]), rr = (int)(key / (uint32_t)G.nc[0]), iy = rr % G.nc[1], iz = rr / G.nc[1];
    float top;
    const int cnt = sor_query(G, q, ix, iy, iz, spts + beg, cell_start + (size_t)s * (kSorCellsCap + 1), K, h, (int)(hq.y & 0xffffu),
                              top);
    dist[vals[hq.x]] = sor_mean_distance(h, cnt, mean_k);
}

// per frame: mean / stddev of the distances -> removal threshold (double).  One CTA per frame, fixed-order tree.
__global__ void __launch_bounds__(kThreads) k_sor_stats(const float* __restrict__ dist, const uint32_t* __restrict__ seg_off,
                                                        double stddev_mul, double* __restrict__ threshold) {
    wait_prior();
    __shared__ double s_sum[kThreads], s_sq[kThreads];
    const int s = blockIdx.x;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    double sum = 0.0, sq = 0.0;
    for (uint32_t i = threadIdx.x; i < n; i += kThreads) {
        const float d = dist[beg + i];
        sum = __dadd_rn(sum, (double)d);
        sq = __dadd_rn(sq, (double)__fmul_rn(d, d));   // PCL: float product
    }
    s_sum[threadIdx.x] = sum; s_sq[threadIdx.x] = sq;
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            s_sum[threadIdx.x] = __dadd_rn(s_sum[threadIdx.x], s_sum[threadIdx.x + o]);
            s_sq[threadIdx.x] = __dadd_rn(s_sq[threadIdx.x], s_sq[threadIdx.x + o]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double nn = (double)n;
        const double mean = __ddiv_rn(s_sum[0], nn);
        const double var = __ddiv_rn(__dsub_rn(s_sq[0], __ddiv_rn(__dmul_rn(s_sum[0], s_sum[0]), nn)), __dsub_rn(nn, 1.0));
        threshold[s] = __dadd_rn(mean, __dmul_rn(stddev_mul, __dsqrt_rn(var)));
    }
}

// stable compaction of the kept points, per frame: counts per tile, then (after a scan) the copy
__global__ void __launch_bounds__(kThreads) k_sor_count(const float* __restrict__ dist, const uint32_t* __restrict__ seg_off,
                                                        const double* __restrict__ threshold, uint32_t tiles_ub,
                                                        uint32_t* __restrict__ tile_cnt) {
    wait_prior();
    __shared__ uint32_t s_c;
    const int s = blockIdx.y;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    if (threadIdx.x == 0) s_c = 0;
    __syncthreads();
    const double thr = threshold[s];
    uint32_t c = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const uint32_t i = blockIdx.x * (kThreads * 4) + threadIdx.x * 4 + r;
        if (i < n && !((double)dist[beg + i] > thr)) ++c;
    }
    c = __reduce_add_sync(kFull, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_c, c);
    __syncthreads();
    if (threadIdx.x == 0) tile_cnt[(size_t)s * tiles_ub + blockIdx.x] = s_c;
}

__global__ void __launch_bounds__(kThreads) k_sor_compact(const float4* __restrict__ pts, const float* __restrict__ dist,
                                                          const uint32_t* __restrict__ seg_off, const double* __restrict__ threshold,
                                                          uint32_t tiles_ub, const uint32_t* __restrict__ tile_off,
                                                          const uint32_t* __restrict__ total, int n_seg,
                                                          float4* __restrict__ out, uint32_t* __restrict__ out_off) {
    wait_prior();
    __shared__ uint32_t s_scan[34];
    const int s = blockIdx.y;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        out_off[s] = tile_off[(size_t)s * tiles_ub];
        if (s == n_seg - 1) out_off[n_seg] = *total;
    }
    const double thr = threshold[s];
    uint32_t flags = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const uint32_t i = blockIdx.x * (kThreads * 4) + threadIdx.x * 4 + r;
        if (i < n && !((double)dist[beg + i] > thr)) flags |= 1u << r;
    }
    uint32_t tot;
    uint32_t o = tile_off[(size_t)s * tiles_ub + blockIdx.x] + block_excl_scan((uint32_t)__popc(flags), s_scan, tot);
#pragma unroll
    for (int r = 0; r < 4; ++r)
        if (flags & (1u << r)) out[o++] = pts[beg + blockIdx.x * (kThreads * 4) + threadIdx.x * 4 + r];
}

}  // namespace o3r
