// voxel.cuh — pcl::VoxelGrid-equivalent downsample on sorted (leaf index, point) pairs.
//
// Engine 1 ("grid"): PCL's own relative 32-bit leaf index per segment (frame), 4-pass radix sort,
//   run detection and a sequential in-order sum per run (CentroidPoint semantics).  Used for the
//   per-frame grid (leaf voxel_size/5), for the one-shot combined grid of RETAIN mode and for the
//   stand-alone o3r_voxel_grid probe.  Because the sort is stable and one thread sums a run in order,
//   centroids are bit-identical to the oracle's, not merely within tolerance.
// Engine 2 ("acc"): the incremental global merge.  64-bit absolute cell keys on the combined grid
//   (leaf v, v, 1000 after z += 500), sort of the cycle's points, and per run a sequential sum that
//   STARTS from the resident accumulator of that cell, so the resident sums equal what a one-shot
//   voxelisation of the whole history would have produced (pose.cpp:434 + :527-531).
#pragma once
#include <type_traits>

#include "common.cuh"
#include "sort.cuh"

namespace o3r {

constexpr int kTileV = kThreads * 4;  // 1024 sorted elements per CTA in the run kernels

// ---- bbox of arbitrary point segments (PCL getMinMax3D), z optionally shifted by +500 ------------------------
// (bbox arrays start as {~0, ~0, ~0, 0, 0, 0} per segment: FILL_BBOX of the host's fill queue)
__global__ void __launch_bounds__(kThreads) k_bbox_pts(const float4* __restrict__ pts, const uint32_t* __restrict__ seg_off,
                                                       int z_shift, uint32_t* __restrict__ bbox) {
    __shared__ uint32_t s_red[6];
    const int s = blockIdx.y;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    if (blockIdx.x * kTileV >= n) return;
    if (threadIdx.x < 6) s_red[threadIdx.x] = (threadIdx.x < 3) ? 0xffffffffu : 0u;
    __syncthreads();
    uint32_t mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t k = blockIdx.x * kTileV + j * kThreads + threadIdx.x;
        if (k < n) {
            const float4 p = pts[beg + k];
            const float z = z_shift ? __fadd_rn(p.z, 500.0f) : p.z;
            const uint32_t ox = f2ord(p.x), oy = f2ord(p.y), oz = f2ord(z);
            mn[0] = min(mn[0], ox); mx[0] = max(mx[0], ox);
            mn[1] = min(mn[1], oy); mx[1] = max(mx[1], oy);
            mn[2] = min(mn[2], oz); mx[2] = max(mx[2], oz);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        mn[a] = __reduce_min_sync(kFull, mn[a]);
        mx[a] = __reduce_max_sync(kFull, mx[a]);
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { atomicMin(&s_red[a], mn[a]); atomicMax(&s_red[3 + a], mx[a]); }
    }
    __syncthreads();
    if (threadIdx.x < 3) atomicMin(&bbox[s * 6 + threadIdx.x], s_red[threadIdx.x]);
    else if (threadIdx.x < 6) atomicMax(&bbox[s * 6 + threadIdx.x], s_red[threadIdx.x]);
}

__global__ void k_grid_params(int n_seg, const uint32_t* __restrict__ bbox, float ix, float iy, float iz,
                              GridParams* __restrict__ grids) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n_seg) grids[s] = make_grid(bbox + 6 * s, ix, iy, iz);
}

// leaf index of arbitrary points (engine 1 when the points do not come from k_emit)
__global__ void __launch_bounds__(kThreads) k_vg_key(const float4* __restrict__ pts, const uint32_t* __restrict__ seg_off,
                                                     const GridParams* __restrict__ grids, int z_shift,
                                                     uint32_t* __restrict__ keys) {
    const int s = blockIdx.y;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    const GridParams G = grids[s];
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        const float4 p = pts[beg + i];
        const float z = z_shift ? __fadd_rn(p.z, 500.0f) : p.z;
        keys[beg + i] = G.passthrough ? i : vg_rel_idx(G, p.x, p.y, z);
    }
}

// ---- engine 1: run heads -> counts; reduce -> centroids ----------------------------------------------------------
struct VgArgs {
    const uint32_t* keys0; const uint32_t* keys1;
    const uint32_t* vals0; const uint32_t* vals1;
    const uint32_t* seg_off;
    const SortPlan* plan;
    const GridParams* grids;     // may be null (no passthrough handling needed beyond keys)
    const float4* pts;
    uint32_t tiles_ub;           // per segment, of kTileV
    uint32_t min_points;
    int z_shift;                 // sums use z + 500 and outputs subtract it again (combined grid)
    float lx_inv, ly_inv, lz_inv;  // for the optional absolute-key output
};

__device__ __forceinline__ bool vg_emits(const uint32_t* keys, uint32_t pos, uint32_t n, uint32_t min_points) {
    if (pos > 0 && keys[pos] == keys[pos - 1]) return false;
    if (min_points <= 1) return true;
    const uint32_t k = keys[pos];
    uint32_t len = 1;
    while (len < min_points && pos + len < n && keys[pos + len] == k) ++len;
    return len >= min_points;
}

__global__ void __launch_bounds__(kThreads) k_vg_heads(VgArgs A, uint32_t* __restrict__ head_cnt) {
    const int s = blockIdx.y;
    const uint32_t t = blockIdx.x;
    const uint32_t beg = A.seg_off[s], n = A.seg_off[s + 1] - beg;
    uint32_t c = 0;
    if (t * kTileV < n) {
        const uint32_t* keys = (A.plan[s].final_parity ? A.keys1 : A.keys0) + beg;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t pos = t * kTileV + threadIdx.x * 4 + j;
            if (pos < n && vg_emits(keys, pos, n, A.min_points)) ++c;
        }
    }
    c = __reduce_add_sync(kFull, c);
    __shared__ uint32_t s_c;
    if (threadIdx.x == 0) s_c = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_c, c);
    __syncthreads();
    if (threadIdx.x == 0) head_cnt[(size_t)s * A.tiles_ub + t] = s_c;
}

__global__ void __launch_bounds__(kThreads) k_vg_reduce(VgArgs A, const uint32_t* __restrict__ head_off,
                                                        const uint32_t* __restrict__ head_total,
                                                        float4* __restrict__ out, uint32_t* __restrict__ seg_out_off,
                                                        int n_seg, uint64_t* __restrict__ out_keys,
                                                        uint32_t* __restrict__ out_counts) {
    __shared__ uint32_t s_scan[34];
    const int s = blockIdx.y;
    const uint32_t t = blockIdx.x;
    if (t == 0 && threadIdx.x == 0) {
        seg_out_off[s] = head_off[(size_t)s * A.tiles_ub];
        if (s == n_seg - 1) seg_out_off[n_seg] = *head_total;
    }
    const uint32_t beg = A.seg_off[s], n = A.seg_off[s + 1] - beg;
    if (t * kTileV >= n) return;
    const int par = A.plan[s].final_parity;
    const bool ident = A.plan[s].n_active == 0;   // nothing was sorted (pass-through / single-cell segment)
    const uint32_t* keys = (par ? A.keys1 : A.keys0) + beg;
    const uint32_t* vals = (par ? A.vals1 : A.vals0) + beg;
    uint32_t flags = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t pos = t * kTileV + threadIdx.x * 4 + j;
        if (pos < n && vg_emits(keys, pos, n, A.min_points)) flags |= 1u << j;
    }
    uint32_t tot;
    uint32_t o = head_off[(size_t)s * A.tiles_ub + t] + block_excl_scan((uint32_t)__popc(flags), s_scan, tot);
    if (!flags) return;
    const bool verbatim = A.grids && A.grids[s].passthrough;  // PCL: output = *input_
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (!(flags & (1u << j))) continue;
        const uint32_t pos = t * kTileV + threadIdx.x * 4 + j;
        const uint32_t k = keys[pos];
        if (verbatim) {
            const float4 p = A.pts[ident ? beg + pos : vals[pos]];
            out[o] = p;
            if (out_keys) out_keys[o] = abs_cell_key(p.x, p.y, A.z_shift ? __fadd_rn(p.z, 500.0f) : p.z, A.lx_inv, A.ly_inv, A.lz_inv);
            if (out_counts) out_counts[o] = 1;
            ++o;
            continue;
        }
        // CentroidPoint<PointXYZRGB>: float sums in run order, divide by (float)n; colour sums as floats
        float sx = 0.f, sy = 0.f, sz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
        uint32_t cnt = 0;
        float4 first = make_float4(0.f, 0.f, 0.f, 0.f);
        for (uint32_t q = pos; q < n && keys[q] == k; ++q) {
            const float4 p = A.pts[ident ? beg + q : vals[q]];
            const float z = A.z_shift ? __fadd_rn(p.z, 500.0f) : p.z;
            if (cnt == 0) first = make_float4(p.x, p.y, z, 0.f);
            const uint32_t c = __float_as_uint(p.w);
            sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, z);
            sr = __fadd_rn(sr, (float)((c >> 16) & 255u));
            sg = __fadd_rn(sg, (float)((c >> 8) & 255u));
            sb = __fadd_rn(sb, (float)(c & 255u));
            ++cnt;
        }
        const float fn = (float)cnt;
        float cz = __fdiv_rn(sz, fn);
        if (A.z_shift) cz = __fsub_rn(cz, 500.0f);
        const uint32_t rgb = ((uint32_t)__fdiv_rn(sr, fn) << 16) | ((uint32_t)__fdiv_rn(sg, fn) << 8) |
                             (uint32_t)__fdiv_rn(sb, fn);
        out[o] = make_float4(__fdiv_rn(sx, fn), __fdiv_rn(sy, fn), cz, __uint_as_float(rgb));
        if (out_keys) out_keys[o] = abs_cell_key(first.x, first.y, first.z, A.lx_inv, A.ly_inv, A.lz_inv);
        if (out_counts) out_counts[o] = cnt;
        ++o;
    }
}

// passthrough segments keep their points verbatim (PCL: output = *input_); the identity keys already make
// every element its own run, so k_vg_reduce reproduces them — except that a centroid of one point is
// sum/1 = the point and uint32(c/1) = c, i.e. bit-identical.  Nothing extra to do.

// ---- CTA-cooperative run reduction (shared by both engines) --------------------------------------------------------
// A CTA owns kTileV consecutive sorted elements.  All threads stage the tile's items into shared memory
// (coalesced key/value loads, gathered item loads), then ONE thread per run adds the run's items strictly in
// sorted (= input) order from shared memory — the oracle's sequential loop, so sums are bit-identical —
// which costs only FADD latency, not memory latency.
// A run that crosses a tile boundary is handed on: the tile where it is still open publishes its partial sums
// (RunCarry, flag last), the next tile's carry thread waits for them, continues with its leading elements and
// either emits the run or hands it on again.  Tiles take their index from an atomic ticket, so the tile being
// waited for is always resident or finished.  Every run is emitted (no min-points filter here).
struct RunCarry {
    float sx, sy, sz;
    uint32_t n, r, g, b, slot, tag, first;   // r, g, b: the policy's colour sums as 32-bit words (col_bits)
    uint32_t pad;
    uint32_t flag;
};  // 48 bytes

// PACKED (point items, weight 1): a = {x, y, z, 0x00RRGGBB}.  Unpacked (partial cells): a = {x, y, z, n}, c = {r, g, b, -}.
template <typename KeyT, bool PACKED>
struct RunSmem {
    float4 a[kTileV];
    uint4 c[PACKED ? 1 : kTileV];
    uint16_t hpos[kTileV + 2];
    uint32_t scan[34];
    uint32_t ticket;
};

// Colour sums: CT = float folds the channels as floats in run order (CentroidPoint, engine 1); CT = uint32_t keeps exact
// integer sums (engine 2's accumulators).  The two agree while a channel sum stays below 2^24.
template <typename CT>
__device__ __forceinline__ void col_add(CT& s, uint32_t v) {
    if constexpr (std::is_same<CT, float>::value) s = __fadd_rn(s, (float)v);
    else s += v;
}
template <typename CT>
__device__ __forceinline__ uint32_t col_bits(CT s) {   // a colour sum as the 32-bit word a RunCarry holds
    if constexpr (std::is_same<CT, float>::value) return __float_as_uint(s);
    else return s;
}
template <typename CT>
__device__ __forceinline__ CT col_from_bits(uint32_t w) {
    if constexpr (std::is_same<CT, float>::value) return __uint_as_float(w);
    else return w;
}

// Sequential sum of staged items [a, e).  Only the FADD chains are serial; the shared-memory loads of the
// next batch are issued before the current batch is added.
template <typename KeyT, bool PACKED, typename CT>
__device__ __forceinline__ void run_sum(const RunSmem<KeyT, PACKED>& S, uint32_t a, uint32_t e, float& sx, float& sy,
                                        float& sz, uint32_t& cn, CT& cr, CT& cg, CT& cb) {
    constexpr int B = 4;
    uint32_t i = a;
    if (PACKED) {
        if (i + B <= e) {
            float4 p[B];
#pragma unroll
            for (int u = 0; u < B; ++u) p[u] = S.a[i + u];
            for (i += B; i + B <= e; i += B) {
                float4 q[B];
#pragma unroll
                for (int u = 0; u < B; ++u) q[u] = S.a[i + u];
#pragma unroll
                for (int u = 0; u < B; ++u) {
                    sx = __fadd_rn(sx, p[u].x); sy = __fadd_rn(sy, p[u].y); sz = __fadd_rn(sz, p[u].z);
                    const uint32_t w = __float_as_uint(p[u].w);
                    col_add(cr, (w >> 16) & 255u); col_add(cg, (w >> 8) & 255u); col_add(cb, w & 255u);
                    p[u] = q[u];
                }
                cn += B;
            }
#pragma unroll
            for (int u = 0; u < B; ++u) {
                sx = __fadd_rn(sx, p[u].x); sy = __fadd_rn(sy, p[u].y); sz = __fadd_rn(sz, p[u].z);
                const uint32_t w = __float_as_uint(p[u].w);
                col_add(cr, (w >> 16) & 255u); col_add(cg, (w >> 8) & 255u); col_add(cb, w & 255u);
            }
            cn += B;
        }
        for (; i < e; ++i) {
            const float4 p = S.a[i];
            sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z);
            const uint32_t w = __float_as_uint(p.w);
            cn += 1; col_add(cr, (w >> 16) & 255u); col_add(cg, (w >> 8) & 255u); col_add(cb, w & 255u);
        }
    } else {
        for (; i + 4 <= e; i += 4) {
            float4 p[4];
            uint4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { p[u] = S.a[i + u]; q[u] = S.c[i + u]; }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                sx = __fadd_rn(sx, p[u].x); sy = __fadd_rn(sy, p[u].y); sz = __fadd_rn(sz, p[u].z);
                cn += __float_as_uint(p[u].w); col_add(cr, q[u].x); col_add(cg, q[u].y); col_add(cb, q[u].z);
            }
        }
        for (; i < e; ++i) {
            const float4 p = S.a[i];
            const uint4 q = S.c[i];
            sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z);
            cn += __float_as_uint(p.w); col_add(cr, q.x); col_add(cg, q.y); col_add(cb, q.z);
        }
    }
}

__device__ __forceinline__ void carry_publish(RunCarry* c, float sx, float sy, float sz, uint32_t n, uint32_t r, uint32_t g,
                                              uint32_t b, uint32_t slot, uint32_t tag, uint32_t first) {
    c->sx = sx; c->sy = sy; c->sz = sz; c->n = n; c->r = r; c->g = g; c->b = b; c->slot = slot; c->tag = tag;
    c->first = first;
    __threadfence();
    st_volatile_u32(&c->flag, 1u);
}

// `carry` points at this tile's RunCarry; carry[-1] is the previous tile of the same segment.
template <typename KeyT, typename Pol>
__device__ __forceinline__ void run_reduce_tile(const KeyT* __restrict__ keys, uint32_t n, uint32_t t, uint32_t slot0,
                                                Pol& pol, RunSmem<KeyT, Pol::kPacked>& S, RunCarry* __restrict__ carry) {
    const int tid = threadIdx.x;
    const uint32_t wbase = t * kTileV;
    const uint32_t wn = min((uint32_t)kTileV, n - wbase);
    // ---- stage the tile
    uint32_t flags = 0;
    {
        const uint32_t p0 = wbase + tid * 4;
        if (p0 + 3 < n) {   // full group: issue the four key/value loads, then the four gathers, then store
            KeyT k4[4];
            const KeyT prev = p0 > 0 ? keys[p0 - 1] : (KeyT)0;
#pragma unroll
            for (int j = 0; j < 4; ++j) k4[j] = keys[p0 + j];
            float4 ia[4];
            uint4 ic[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pol.load(p0 + j, ia[j], ic[j]);
            if (p0 == 0 || k4[0] != prev) flags |= 1u;
#pragma unroll
            for (int j = 1; j < 4; ++j)
                if (k4[j] != k4[j - 1]) flags |= 1u << j;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                S.a[tid * 4 + j] = ia[j];
                if (!Pol::kPacked) S.c[tid * 4 + j] = ic[j];
            }
        } else {
            KeyT prev = (p0 > 0 && p0 < n) ? keys[p0 - 1] : (KeyT)0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t pos = p0 + j;
                if (pos < n) {
                    const KeyT key = keys[pos];
                    if (pos == 0 || key != prev) flags |= 1u << j;
                    prev = key;
                    const int e = tid * 4 + j;
                    float4 ia; uint4 ic;
                    pol.load(pos, ia, ic);
                    S.a[e] = ia;
                    if (!Pol::kPacked) S.c[e] = ic;
                }
            }
        }
    }
    uint32_t H;
    uint32_t hoff = block_excl_scan((uint32_t)__popc(flags), S.scan, H);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (flags & (1u << j)) S.hpos[hoff++] = (uint16_t)(tid * 4 + j);
    if (tid == 0) S.hpos[H] = (uint16_t)wn;
    __syncthreads();
    const bool more = wbase + wn < n;              // the segment continues after this tile
    // ---- one thread per run whose head lies in the tile
    for (uint32_t rI = tid; rI < H; rI += kThreads) {
        const uint32_t a = S.hpos[rI], e = S.hpos[rI + 1];
        const bool tail = rI == H - 1 && more;
        const KeyT key = (Pol::kNeedsKey || tail) ? keys[wbase + a] : (KeyT)0;
        float sx = 0.f, sy = 0.f, sz = 0.f;
        uint32_t cn = 0, tag = 0;
        typename Pol::ColT cr = 0, cg = 0, cb = 0;
        pol.start(wbase + a, sx, sy, sz, cn, cr, cg, cb, tag);
        const uint32_t first_v = wbase + a;   // position of the run's first element
        run_sum(S, a, e, sx, sy, sz, cn, cr, cg, cb);
        if (tail && keys[wbase + wn] == key)   // still open at the tile end: hand it on
            carry_publish(carry, sx, sy, sz, cn, col_bits(cr), col_bits(cg), col_bits(cb), slot0 + rI, tag, first_v);
        else
            pol.emit(slot0 + rI, key, sx, sy, sz, cn, cr, cg, cb, tag, first_v);
    }
    // ---- the run handed over by the previous tile: its elements are the tile's leading ones
    const uint32_t lead = H ? S.hpos[0] : wn;
    if (tid == kThreads - 1 && lead > 0) {
        const RunCarry* pc = carry - 1;
        while (ld_volatile_u32(&pc->flag) == 0u) __nanosleep(64);
        __threadfence();
        float sx = __ldcg(&pc->sx), sy = __ldcg(&pc->sy), sz = __ldcg(&pc->sz);
        uint32_t cn = __ldcg(&pc->n);
        using CT = typename Pol::ColT;
        CT cr = col_from_bits<CT>(__ldcg(&pc->r)), cg = col_from_bits<CT>(__ldcg(&pc->g)), cb = col_from_bits<CT>(__ldcg(&pc->b));
        const uint32_t slot = __ldcg(&pc->slot), tag = __ldcg(&pc->tag), first_v = __ldcg(&pc->first);
        run_sum(S, 0u, lead, sx, sy, sz, cn, cr, cg, cb);
        const KeyT key = keys[wbase];
        if (H == 0 && more && keys[wbase + wn] == key)
            carry_publish(carry, sx, sy, sz, cn, col_bits(cr), col_bits(cg), col_bits(cb), slot, tag, first_v);
        else
            pol.emit(slot, key, sx, sy, sz, cn, cr, cg, cb, tag, first_v);
    }
}

// engine 1 policy: CentroidPoint of a VoxelGrid leaf (coordinate and colour channels folded as floats in run order, as
// k_vg_reduce and PCL do).  Optionally tracks the range of combined-grid cells the emitted centroids fall in (so the
// merge can sort compact keys).
struct VgPol {
    static constexpr bool kNeedsKey = false;
    static constexpr bool kPacked = true;
    using ColT = float;
    const float4* spts;   // the segment's points when they are already in sorted order (null: gather pts[vals[pos]])
    const float4* pts; const uint32_t* vals;
    float4* out; int z_shift; bool verbatim;
    int want_cells; float icx, icz;
    int mn[3], mx[3];
    __device__ __forceinline__ void load(uint32_t pos, float4& a, uint4&) const {
        a = spts ? __ldcs(spts + pos) : pts[vals[pos]];
        if (z_shift) a.z = __fadd_rn(a.z, 500.0f);
    }
    __device__ __forceinline__ void start(uint32_t, float&, float&, float&, uint32_t&, float&, float&, float&,
                                          uint32_t&) const {}   // sums start at zero
    __device__ __forceinline__ void emit(uint32_t slot, uint32_t, float sx, float sy, float sz, uint32_t n, float r,
                                         float g, float b, uint32_t, uint32_t first) {
        float4 o;
        if (verbatim) {   // PCL: output = *input_
            o = spts ? spts[first] : pts[vals[first]];
        } else {
            const float fn = (float)n;
            float cz = __fdiv_rn(sz, fn);
            if (z_shift) cz = __fsub_rn(cz, 500.0f);
            const uint32_t rgb = ((uint32_t)__fdiv_rn(r, fn) << 16) | ((uint32_t)__fdiv_rn(g, fn) << 8) |
                                 (uint32_t)__fdiv_rn(b, fn);
            o = make_float4(__fdiv_rn(sx, fn), __fdiv_rn(sy, fn), cz, __uint_as_float(rgb));
        }
        out[slot] = o;
        if (want_cells) {
            const int ci = (int)floorf(__fmul_rn(o.x, icx)), cj = (int)floorf(__fmul_rn(o.y, icx)),
                      ck = (int)floorf(__fmul_rn(__fadd_rn(o.z, 500.0f), icz));
            mn[0] = min(mn[0], ci); mx[0] = max(mx[0], ci);
            mn[1] = min(mn[1], cj); mx[1] = max(mx[1], cj);
            mn[2] = min(mn[2], ck); mx[2] = max(mx[2], ck);
        }
    }
};

// fast path of engine 1: every run is emitted (min_points <= 1), no key / count outputs.
// Linear grid of tiles_ub * n_seg CTAs; work[0] is the ticket, carries follow.
#ifndef O3R_VG_MINB
#define O3R_VG_MINB 5
#endif
__global__ void __launch_bounds__(kThreads, O3R_VG_MINB) k_vg_reduce_w(VgArgs A, const uint32_t* __restrict__ head_off,
                                                          const uint32_t* __restrict__ head_total,
                                                          float4* __restrict__ out, uint32_t* __restrict__ seg_out_off,
                                                          int n_seg, uint32_t* __restrict__ ticket,
                                                          RunCarry* __restrict__ carries, int want_cells, float icx,
                                                          float icz, int* __restrict__ cellbb,
                                                          const uint32_t* __restrict__ out_base) {
    __shared__ RunSmem<uint32_t, true> S;
    __shared__ int s_bb[6];
    if (threadIdx.x == 0) S.ticket = atomicAdd(ticket, 1u);
    if (threadIdx.x < 6) s_bb[threadIdx.x] = threadIdx.x < 3 ? 0x7fffffff : (int)0x80000000;
    __syncthreads();
    const uint32_t lin = S.ticket;
    const int s = lin / A.tiles_ub;
    const uint32_t t = lin - (uint32_t)s * A.tiles_ub;
    const uint32_t obase = out_base ? *out_base : 0u;   // batch-wide output position of this chunk
    if (t == 0 && threadIdx.x == 0) {
        seg_out_off[s] = obase + head_off[(size_t)s * A.tiles_ub];
        if (s == n_seg - 1 && !out_base) seg_out_off[n_seg] = *head_total;
    }
    const uint32_t beg = A.seg_off[s], n = A.seg_off[s + 1] - beg;
    if (t * kTileV >= n) return;
    const SortPlan pl = A.plan[s];
    const int par = pl.final_parity;
    // a segment that needed no radix pass is already in order: its points are read sequentially, not gathered
    const float4* sp = pl.n_active ? nullptr : A.pts + beg;
    VgPol pol{sp, A.pts, (par ? A.vals1 : A.vals0) + beg, out + obase, A.z_shift, A.grids && A.grids[s].passthrough,
              want_cells, icx, icz,
              {0x7fffffff, 0x7fffffff, 0x7fffffff}, {(int)0x80000000, (int)0x80000000, (int)0x80000000}};
    run_reduce_tile<uint32_t, VgPol>((par ? A.keys1 : A.keys0) + beg, n, t, head_off[(size_t)s * A.tiles_ub + t], pol, S,
                                     carries + lin);
    if (want_cells) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const int lo = __reduce_min_sync(kFull, pol.mn[a]), hi = __reduce_max_sync(kFull, pol.mx[a]);
            if ((threadIdx.x & 31) == 0) { atomicMin(&s_bb[a], lo); atomicMax(&s_bb[3 + a], hi); }
        }
        __syncthreads();
        if (threadIdx.x < 3) atomicMin(&cellbb[threadIdx.x], s_bb[threadIdx.x]);
        else if (threadIdx.x < 6) atomicMax(&cellbb[threadIdx.x], s_bb[threadIdx.x]);
    }
}

// ---- engine 2: incremental merge on the combined grid -----------------------------------------------------------
// The cycle's items are sorted by a COMPACT key: cell coordinates relative to the cycle's minimum cell, packed
// (k | j | i) into just the bits the cycle's extent needs (3 radix passes instead of 6-8 on the absolute key).
// Field-wise subtraction of a constant keeps the (k, j, i) lexicographic order, so the sorted cycle list is in
// the same order as the resident shard, which stores the absolute key.
struct KeyCodec {
    int imin, jmin, kmin;
    int wi, wj;           // bit widths of the i and j fields
    __device__ __forceinline__ uint64_t pack(int i, int j, int k) const {
        return ((uint64_t)(uint32_t)(k - kmin) << (wi + wj)) | ((uint64_t)(uint32_t)(j - jmin) << wi) |
               (uint64_t)(uint32_t)(i - imin);
    }
    __device__ __forceinline__ uint64_t to_abs(uint64_t c) const {
        const long long B = 1 << 20;
        const long long i = (long long)(c & ((1ull << wi) - 1ull)) + imin;
        const long long j = (long long)((c >> wi) & ((1ull << wj) - 1ull)) + jmin;
        const long long k = (long long)(c >> (wi + wj)) + kmin;
        return ((uint64_t)(k + B) << 42) | ((uint64_t)(j + B) << 21) | (uint64_t)(i + B);
    }
};

struct AccItemsPts {   // items are points of weight 1 (z gets +500)
    const float4* pts;
    const float4* spts;    // the points themselves when nothing had to be sorted (already in order), else null
    const uint32_t* vals;  // sorted order -> point index (when spts is null)
    static constexpr bool kGather = true;
    static constexpr bool kPacked = true;
    __device__ __forceinline__ void get(uint32_t pos, float4& a, uint4&) const {
        a = spts ? __ldcs(spts + pos) : pts[vals[pos]];
        a.z = __fadd_rn(a.z, 500.0f);
    }
    __device__ __forceinline__ void cell(uint32_t v, float ix, float iz, int& i, int& j, int& k) const {
        const float4 p = pts[v];
        i = (int)floorf(__fmul_rn(p.x, ix)); j = (int)floorf(__fmul_rn(p.y, ix));
        k = (int)floorf(__fmul_rn(__fadd_rn(p.z, 500.0f), iz));
    }
    __device__ __forceinline__ bool finite(uint32_t v) const {
        const float4 p = pts[v];
        return isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    }
};
struct AccItemsCells {  // items are partial cells received from other ranks
    const o3r_cell* cells;
    const float4* spts;    // unused
    const uint32_t* vals;  // sorted order -> cell index
    static constexpr bool kGather = false;
    static constexpr bool kPacked = false;
    __device__ __forceinline__ void get(uint32_t pos, float4& a, uint4& q) const {
        const o3r_cell c = cells[vals[pos]];
        a = make_float4(c.sx, c.sy, c.sz, __uint_as_float(c.n));
        q = make_uint4(c.sr, c.sg, c.sb, 0u);
    }
    __device__ __forceinline__ void cell(uint32_t v, float, float, int& i, int& j, int& k) const {
        const uint64_t key = cells[v].key;
        const int B = 1 << 20;
        i = (int)(key & 0x1fffffu) - B; j = (int)((key >> 21) & 0x1fffffu) - B; k = (int)(key >> 42) - B;
    }
    __device__ __forceinline__ bool finite(uint32_t) const { return true; }
};

// range of combined-grid cells of n items (only when the range was not tracked upstream).  A NaN coordinate converts to
// cell 0, so a non-finite item widens the range to INT_MIN instead, which the host refuses like any cell beyond +-2^20.
template <typename Items>
__global__ void __launch_bounds__(kThreads) k_acc_cellbb(Items items, uint32_t n, float ix, float iz, int* __restrict__ cellbb) {
    int mn[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff}, mx[3] = {(int)0x80000000, (int)0x80000000, (int)0x80000000};
    for (uint32_t v = blockIdx.x * kThreads + threadIdx.x; v < n; v += gridDim.x * kThreads) {
        int c[3];
        items.cell(v, ix, iz, c[0], c[1], c[2]);
        if (!items.finite(v)) c[0] = (int)0x80000000;
#pragma unroll
        for (int a = 0; a < 3; ++a) { mn[a] = min(mn[a], c[a]); mx[a] = max(mx[a], c[a]); }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int lo = __reduce_min_sync(kFull, mn[a]), hi = __reduce_max_sync(kFull, mx[a]);
        if ((threadIdx.x & 31) == 0) { atomicMin(&cellbb[a], lo); atomicMax(&cellbb[3 + a], hi); }
    }
}

// after a chunk: advance the batch-wide output position and record it as the next frame's offset
__global__ void k_add_base(uint32_t* base, const uint32_t* total, uint32_t* goff_end) {
    if (threadIdx.x == 0) { *base += *total; *goff_end = *base; }
}

// compact keys of the cycle's items + whole-array digit histograms for the plan's digit layout
template <typename KeyT, typename Items>
__global__ void __launch_bounds__(kThreads) k_acc_key(Items items, uint32_t n, float ix, float iz, KeyCodec kc,
                                                      const SortPlan* __restrict__ plan, KeyT* __restrict__ keys,
                                                      uint32_t* __restrict__ vals, uint32_t* __restrict__ ghist,
                                                      const uint32_t* __restrict__ n_dev, uint32_t* __restrict__ seg_out) {
    __shared__ uint32_t sh[kMaxPasses * kRsBins];
    if (n_dev) {   // the item count lives on the device (n is the host's bound); publish the segment for the sort
        n = min(n, *n_dev);
        if (blockIdx.x == 0 && threadIdx.x == 0) { seg_out[0] = 0u; seg_out[1] = n; }
    }
    const int np = plan[0].n_passes;
    for (int i = threadIdx.x; i < np * kRsBins; i += kThreads) sh[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (uint32_t base = blockIdx.x * kThreads; base < n; base += gridDim.x * kThreads) {
        const uint32_t v = base + threadIdx.x;
        const bool valid = v < n;
        KeyT k = 0;
        if (valid) {
            int ci, cj, ck;
            items.cell(v, ix, iz, ci, cj, ck);
            k = (KeyT)kc.pack(ci, cj, ck);
            keys[v] = k;
            vals[v] = v;
        }
        const unsigned vm = __ballot_sync(kFull, valid);
        if (valid)
            for (int p = 0; p < np; ++p)
                hist_add(sh + p * kRsBins, rs_digit(k, (int)plan[0].shift[p], (1u << plan[0].bits[p]) - 1u), vm, lane);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < np * kRsBins; i += kThreads)
        if (sh[i]) atomicAdd(&ghist[i], sh[i]);
}

template <typename KeyT>
struct AccArgs {
    const KeyT* keys0; const KeyT* keys1;
    const uint32_t* vals0; const uint32_t* vals1;
    const uint32_t* seg_off;      // [2] = {0, n}
    const SortPlan* plan;         // [1]
    uint32_t tiles_ub;
    KeyCodec kc;
    // resident shard (sorted by absolute key)
    const uint64_t* res_keys; float4* res_acc; uint4* res_rgb;
    const uint32_t* n_res_ptr;    // resident cell count lives on the device (the merge never syncs with the host)
};

// Counts the run heads of each tile and — fully in parallel, one thread per head — looks every head's cell up in
// the resident shard.  The result (position + 1, or 0 for a new cell) is parked at the head's element position in
// the ping-pong value buffer the sort left idle, where k_acc_reduce picks it up.
template <typename KeyT>
__global__ void __launch_bounds__(kThreads) k_acc_heads(AccArgs<KeyT> A, uint32_t* __restrict__ vals0, uint32_t* __restrict__ vals1,
                                                        uint32_t* __restrict__ head_cnt, uint32_t* __restrict__ n_new) {
    const uint32_t t = blockIdx.x;
    const uint32_t n = A.seg_off[1];
    uint32_t c = 0, fresh = 0;
    if (t * kTileV < n) {
        const int par = A.plan[0].final_parity;
        const KeyT* keys = par ? A.keys1 : A.keys0;
        uint32_t* tags = par ? vals0 : vals1;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t pos = t * kTileV + j * kThreads + threadIdx.x;   // coalesced
            if (pos < n) {
                const KeyT ck = keys[pos];
                if (pos == 0 || ck != keys[pos - 1]) {
                    ++c;
                    const uint64_t k = A.kc.to_abs((uint64_t)ck);
                    const uint32_t n_res = *A.n_res_ptr;
                    uint32_t lo = 0, hi = n_res;  // lower_bound in the resident keys
                    while (lo < hi) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if (A.res_keys[mid] < k) lo = mid + 1; else hi = mid;
                    }
                    const bool found = lo < n_res && A.res_keys[lo] == k;
                    tags[pos] = found ? lo + 1 : 0u;
                    if (!found) ++fresh;
                }
            }
        }
    }
    c = __reduce_add_sync(kFull, c);
    fresh = __reduce_add_sync(kFull, fresh);
    __shared__ uint32_t s_c, s_f;
    if (threadIdx.x == 0) { s_c = 0; s_f = 0; }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { if (c) atomicAdd(&s_c, c); if (fresh) atomicAdd(&s_f, fresh); }
    __syncthreads();
    if (threadIdx.x == 0) { head_cnt[t] = s_c; if (s_f) atomicAdd(n_new, s_f); }
}

// engine 2 policy: look the cell up in the resident shard and continue its sums in input order.
// Emits the cycle's cell list (sorted by key): ckey (absolute), cacc = {sx, sy, sz, n}, crgb = {sr, sg, sb, found_pos + 1}.
// Colour sums are exact uint32 (they differ from a float fold once a channel sum passes 2^24; DESIGN §2).
template <typename KeyT, typename Items>
struct AccPol {
    static constexpr bool kNeedsKey = true;
    static constexpr bool kPacked = Items::kPacked;
    using ColT = uint32_t;
    Items items;
    KeyCodec kc;
    const uint32_t* tags;   // per element position: resident position + 1 of a head's cell, 0 = new cell
    const float4* res_acc; const uint4* res_rgb;
    uint64_t* ckey; float4* cacc; uint4* crgb;
    __device__ __forceinline__ void load(uint32_t pos, float4& a, uint4& c) const { items.get(pos, a, c); }
    __device__ __forceinline__ void start(uint32_t pos, float& sx, float& sy, float& sz, uint32_t& n, uint32_t& r,
                                          uint32_t& g, uint32_t& b, uint32_t& tag) const {
        tag = tags[pos];
        if (tag) {
            const float4 a = res_acc[tag - 1];
            const uint4 c = res_rgb[tag - 1];
            sx = a.x; sy = a.y; sz = a.z; n = __float_as_uint(a.w); r = c.x; g = c.y; b = c.z;
        }
    }
    __device__ __forceinline__ void emit(uint32_t slot, KeyT ck, float sx, float sy, float sz, uint32_t n, uint32_t r,
                                         uint32_t g, uint32_t b, uint32_t tag, uint32_t) const {
        ckey[slot] = kc.to_abs((uint64_t)ck);
        cacc[slot] = make_float4(sx, sy, sz, __uint_as_float(n));
        crgb[slot] = make_uint4(r, g, b, tag);
    }
};

template <typename KeyT, typename Items>
__global__ void __launch_bounds__(kThreads, 5) k_acc_reduce(AccArgs<KeyT> A, Items items, const uint32_t* __restrict__ head_off,
                                                         uint64_t* __restrict__ ckey, float4* __restrict__ cacc,
                                                         uint4* __restrict__ crgb, uint32_t* __restrict__ ticket,
                                                         RunCarry* __restrict__ carries) {
    __shared__ RunSmem<KeyT, Items::kPacked> S;
    if (threadIdx.x == 0) S.ticket = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t t = S.ticket;
    const uint32_t n = A.seg_off[1];
    if (t * kTileV >= n) return;
    const SortPlan pl = A.plan[0];
    const int par = pl.final_parity;
    items.vals = par ? A.vals1 : A.vals0;
    if constexpr (Items::kGather) { if (!pl.n_active) items.spts = items.pts; }   // nothing was sorted: already in order
    AccPol<KeyT, Items> pol{items, A.kc, par ? A.vals0 : A.vals1, A.res_acc, A.res_rgb, ckey, cacc, crgb};
    run_reduce_tile<KeyT, AccPol<KeyT, Items>>(par ? A.keys1 : A.keys0, n, t, head_off[t], pol, S, carries + t);
}

// found cells: write the continued sums back in place; new cells: flag for compaction
// (launched over an upper bound of the cycle's cell count; the exact count is read from the device)
__global__ void __launch_bounds__(kThreads) k_acc_update(const uint32_t* __restrict__ n_cyc_ptr, const float4* __restrict__ cacc,
                                                         const uint4* __restrict__ crgb, float4* __restrict__ res_acc,
                                                         uint4* __restrict__ res_rgb, uint32_t* __restrict__ new_cnt) {
    const uint32_t n_cyc = *n_cyc_ptr;
    const uint32_t t = blockIdx.x;
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t h = t * kTileV + threadIdx.x * 4 + j;
        if (h < n_cyc) {
            const uint4 r = crgb[h];
            if (r.w) {
                res_acc[r.w - 1] = cacc[h];
                res_rgb[r.w - 1] = make_uint4(r.x, r.y, r.z, 0u);
            } else {
                ++c;
            }
        }
    }
    c = __reduce_add_sync(kFull, c);
    __shared__ uint32_t s_c;
    if (threadIdx.x == 0) s_c = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_c, c);
    __syncthreads();
    if (threadIdx.x == 0) new_cnt[t] = s_c;
}

// new cells go to their merged position: q-th new cell -> q + lower_bound(res_keys, key)
__global__ void __launch_bounds__(kThreads) k_acc_place_new(const uint32_t* __restrict__ n_cyc_ptr, const uint64_t* __restrict__ ckey,
                                                            const float4* __restrict__ cacc, const uint4* __restrict__ crgb,
                                                            const uint32_t* __restrict__ new_off,
                                                            const uint64_t* __restrict__ res_keys,
                                                            const uint32_t* __restrict__ n_res_ptr,
                                                            uint64_t* __restrict__ dst_keys, float4* __restrict__ dst_acc,
                                                            uint4* __restrict__ dst_rgb, uint64_t* __restrict__ new_keys) {
    __shared__ uint32_t s_scan[34];
    const uint32_t n_cyc = *n_cyc_ptr, n_res = *n_res_ptr;
    const uint32_t t = blockIdx.x;
    if (t * kTileV >= n_cyc) return;
    uint32_t flags = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t h = t * kTileV + threadIdx.x * 4 + j;
        if (h < n_cyc && crgb[h].w == 0) flags |= 1u << j;
    }
    uint32_t tot;
    uint32_t q = new_off[t] + block_excl_scan((uint32_t)__popc(flags), s_scan, tot);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (!(flags & (1u << j))) continue;
        const uint32_t h = t * kTileV + threadIdx.x * 4 + j;
        const uint64_t k = ckey[h];
        uint32_t lo = 0, hi = n_res;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (res_keys[mid] < k) lo = mid + 1; else hi = mid;
        }
        const uint32_t d = q + lo;
        dst_keys[d] = k;
        dst_acc[d] = cacc[h];
        const uint4 r = crgb[h];
        dst_rgb[d] = make_uint4(r.x, r.y, r.z, 0u);
        new_keys[q] = k;
        ++q;
    }
}

// resident cells shift right by the number of new cells with a smaller key
__global__ void __launch_bounds__(kThreads) k_acc_place_old(const uint32_t* __restrict__ n_res_ptr,
                                                            const uint64_t* __restrict__ res_keys,
                                                            const float4* __restrict__ res_acc, const uint4* __restrict__ res_rgb,
                                                            const uint64_t* __restrict__ new_keys,
                                                            const uint32_t* __restrict__ n_new_ptr,
                                                            uint64_t* __restrict__ dst_keys, float4* __restrict__ dst_acc,
                                                            uint4* __restrict__ dst_rgb) {
    const uint32_t n_res = *n_res_ptr, n_new = *n_new_ptr;
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n_res; i += gridDim.x * kThreads) {
        const uint64_t k = res_keys[i];
        uint32_t lo = 0, hi = n_new;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (new_keys[mid] < k) lo = mid + 1; else hi = mid;
        }
        const uint32_t d = i + lo;
        dst_keys[d] = k;
        dst_acc[d] = res_acc[i];
        dst_rgb[d] = res_rgb[i];
    }
}

// the merged shard now holds n_res + n_new cells
__global__ void k_acc_finish(uint32_t* n_res, const uint32_t* n_new) {
    if (threadIdx.x == 0) *n_res += *n_new;
}

// downsamplePtCloud(cloud_big, true) on the accumulators: count >= min_points -> centroid, z -= 500
// (launched over an upper bound of the resident cell count; the exact count is read from the device)
__global__ void __launch_bounds__(kThreads) k_acc_emit_cnt(const uint32_t* __restrict__ n_res_ptr, const float4* __restrict__ res_acc,
                                                           uint32_t min_points, uint32_t* __restrict__ cnt) {
    const uint32_t n_res = *n_res_ptr;
    const uint32_t t = blockIdx.x;
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t i = t * kTileV + threadIdx.x * 4 + j;
        if (i < n_res && __float_as_uint(res_acc[i].w) >= min_points) ++c;
    }
    c = __reduce_add_sync(kFull, c);
    __shared__ uint32_t s_c;
    if (threadIdx.x == 0) s_c = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_c, c);
    __syncthreads();
    if (threadIdx.x == 0) cnt[t] = s_c;
}

// one cell's output record from its accumulators {sx, sy, sz + 500, n} and colour sums: the one place this arithmetic lives
// (k_acc_emit and the change set's k_chg_emit both call it, so their records cannot drift apart)
__device__ __forceinline__ float4 acc_centroid(const float4 a, const uint4 c) {
    const float fn = (float)__float_as_uint(a.w);
    const uint32_t rgb = ((uint32_t)__fdiv_rn((float)c.x, fn) << 16) | ((uint32_t)__fdiv_rn((float)c.y, fn) << 8) |
                         (uint32_t)__fdiv_rn((float)c.z, fn);
    return make_float4(__fdiv_rn(a.x, fn), __fdiv_rn(a.y, fn), __fsub_rn(__fdiv_rn(a.z, fn), 500.0f), __uint_as_float(rgb));
}

__global__ void __launch_bounds__(kThreads) k_acc_emit(const uint32_t* __restrict__ n_res_ptr, const float4* __restrict__ res_acc,
                                                       const uint4* __restrict__ res_rgb, uint32_t min_points,
                                                       const uint32_t* __restrict__ off, float4* __restrict__ out) {
    __shared__ uint32_t s_scan[34];
    const uint32_t n_res = *n_res_ptr;
    const uint32_t t = blockIdx.x;
    uint32_t flags = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t i = t * kTileV + threadIdx.x * 4 + j;
        if (i < n_res && __float_as_uint(res_acc[i].w) >= min_points) flags |= 1u << j;
    }
    uint32_t tot;
    uint32_t o = off[t] + block_excl_scan((uint32_t)__popc(flags), s_scan, tot);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (!(flags & (1u << j))) continue;
        const uint32_t i = t * kTileV + threadIdx.x * 4 + j;
        out[o++] = acc_centroid(res_acc[i], res_rgb[i]);
    }
}

// ---- multi-GPU exchange helpers -------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t hash64(uint64_t x) {  // splitmix64 finaliser
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27; x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

// owner of each cycle cell + per-owner histogram; keys32 = owner, vals = cell index (then one sort pass)
// (the cell count is read from the device; seg receives {0, n_cyc} for the sort that follows)
__global__ void __launch_bounds__(kThreads) k_owner(const uint32_t* __restrict__ n_cyc_ptr, const uint64_t* __restrict__ ckey,
                                                    uint32_t world, uint32_t* __restrict__ okeys, uint32_t* __restrict__ ovals,
                                                    uint32_t* __restrict__ counts, uint32_t* __restrict__ seg) {
    __shared__ uint32_t s_cnt[256];   // (world <= 256) the CTA's histogram: one global atomic per owner and CTA, not per cell
    const uint32_t n_cyc = *n_cyc_ptr;
    if (blockIdx.x == 0 && threadIdx.x == 0) { seg[0] = 0u; seg[1] = n_cyc; }
    for (uint32_t r = threadIdx.x; r < world; r += kThreads) s_cnt[r] = 0u;
    __syncthreads();
    const uint32_t n_round = (n_cyc + 31u) & ~31u;   // whole warps take every trip (match_any below)
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n_round; i += gridDim.x * kThreads) {
        uint32_t o = 0xffffffffu;
        if (i < n_cyc) {
            o = (uint32_t)(hash64(ckey[i]) % world);
            okeys[i] = o;
            ovals[i] = i;
        }
        const unsigned peers = __match_any_sync(kFull, o);
        if (o != 0xffffffffu && (peers & ((1u << (threadIdx.x & 31)) - 1u)) == 0u) atomicAdd(&s_cnt[o], (uint32_t)__popc(peers));
    }
    __syncthreads();
    for (uint32_t r = threadIdx.x; r < world; r += kThreads)
        if (s_cnt[r]) atomicAdd(&counts[r], s_cnt[r]);
}

// rigid transform of a resident point cloud in place (pose.cpp:353)
__global__ void __launch_bounds__(kThreads) k_transform_pts(float4* __restrict__ pts, size_t n, const float* __restrict__ Tm) {
    __shared__ float T[12];
    if (threadIdx.x < 12) T[threadIdx.x] = Tm[threadIdx.x];
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        float4 p = pts[i];
        float x, y, z;
        xform(T, p.x, p.y, p.z, x, y, z);
        p.x = x; p.y = y; p.z = z;
        pts[i] = p;
    }
}

}  // namespace o3r
