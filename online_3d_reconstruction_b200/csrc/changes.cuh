// changes.cuh — change tracking of the resident cloud (accumulate modes): the pending set D of cells whose point count grew
// since the consumer last read the changes, and the emission of those cells' records.
//
// D is a sorted, unique list of absolute 63-bit cell keys.  Every merged cycle unites it with the cycle's distinct cells
// (ckey[0 .. counters[CNT_CYC]), sorted by the same key) by a merge-path set union: k_chg_part splits the merged sequence
// into tiles of kTileV elements, k_chg_union<false> counts each tile's unique elements, k_scan_u32 turns the counts into
// offsets (and the total into D's new count), k_chg_union<true> writes.  In merged order an element equal to its predecessor
// is a duplicate (both lists are unique, so a cell present in both appears twice, adjacent).  Launches are sized by host
// upper bounds; every kernel reads the exact list lengths from device memory.
#pragma once
#include "voxel.cuh"

namespace o3r {

constexpr uint32_t kChgNone = 0xffffffffu;

// merge path: how many elements of a come first among the first d elements of merge(a, b) (ties: a first)
__device__ __forceinline__ uint32_t merge_path(const uint64_t* a, uint32_t na, const uint64_t* b, uint32_t nb, uint32_t d) {
    uint32_t lo = d > nb ? d - nb : 0u, hi = d < na ? d : na;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] <= b[d - mid - 1]) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// part[t] = elements of a before diagonal t * kTileV (t = 0 .. tiles)
__global__ void __launch_bounds__(kThreads) k_chg_part(const uint64_t* __restrict__ a, const uint32_t* __restrict__ na_ptr,
                                                       const uint64_t* __restrict__ b, const uint32_t* __restrict__ nb_ptr,
                                                       uint32_t tiles, uint32_t* __restrict__ part) {
    wait_prior();
    const uint32_t t = blockIdx.x * kThreads + threadIdx.x;
    if (t > tiles) return;
    const uint32_t na = *na_ptr, nb = *nb_ptr;
    const uint64_t d = min((uint64_t)t * kTileV, (uint64_t)na + nb);
    part[t] = merge_path(a, na, b, nb, (uint32_t)d);
}

// One tile of merge(a, b) per CTA, 4 consecutive merged elements per thread.  kWrite = false: cnt[t] = the tile's unique
// elements; kWrite = true: writes them to out at off[t].
template <bool kWrite>
__global__ void __launch_bounds__(kThreads) k_chg_union(const uint64_t* __restrict__ a, const uint32_t* __restrict__ na_ptr,
                                                        const uint64_t* __restrict__ b, const uint32_t* __restrict__ nb_ptr,
                                                        const uint32_t* __restrict__ part, uint32_t* __restrict__ cnt,
                                                        const uint32_t* __restrict__ off, uint64_t* __restrict__ out) {
    wait_prior();
    __shared__ uint64_t s_a[kTileV], s_b[kTileV];
    __shared__ uint32_t s_scan[34];
    const uint32_t na = *na_ptr, nb = *nb_ptr, n = na + nb;
    const uint32_t t = blockIdx.x;
    const uint32_t d0 = t * kTileV;
    if (d0 >= n) {
        if (!kWrite && threadIdx.x == 0) cnt[t] = 0u;
        return;
    }
    const uint32_t d1 = (uint32_t)min((uint64_t)d0 + kTileV, (uint64_t)n);
    const uint32_t a0 = part[t], a1 = part[t + 1], b0 = d0 - a0, b1 = d1 - a1;
    const uint32_t ta = a1 - a0, tb = b1 - b0;
    for (uint32_t i = threadIdx.x; i < ta; i += kThreads) s_a[i] = a[a0 + i];
    for (uint32_t i = threadIdx.x; i < tb; i += kThreads) s_b[i] = b[b0 + i];
    // the element just before the tile in merged order: the larger of the two lists' last elements before the diagonal
    bool have_prev = false;
    uint64_t tile_prev = 0;
    if (a0) { tile_prev = a[a0 - 1]; have_prev = true; }
    if (b0) { const uint64_t v = b[b0 - 1]; tile_prev = have_prev ? max(tile_prev, v) : v; have_prev = true; }
    __syncthreads();
    const uint32_t ld = min((uint32_t)threadIdx.x * 4u, ta + tb);
    uint32_t ia = merge_path(s_a, ta, s_b, tb, ld), ib = ld - ia;
    uint64_t prev = tile_prev;
    bool hp = have_prev;
    if (ia || ib) {   // the merged element at ld - 1
        hp = true;
        prev = ia ? s_a[ia - 1] : s_b[ib - 1];
        if (ia && ib) prev = max(s_a[ia - 1], s_b[ib - 1]);
    }
    uint64_t v[4] = {0, 0, 0, 0};
    uint32_t flags = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (ld + j >= ta + tb) break;
        const bool take_a = ia < ta && (ib >= tb || s_a[ia] <= s_b[ib]);
        v[j] = take_a ? s_a[ia++] : s_b[ib++];
        if (!hp || v[j] != prev) flags |= 1u << j;
        prev = v[j];
        hp = true;
    }
    if (!kWrite) {
        uint32_t c = __reduce_add_sync(kFull, (uint32_t)__popc(flags));
        __shared__ uint32_t s_c;
        if (threadIdx.x == 0) s_c = 0;
        __syncthreads();
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_c, c);
        __syncthreads();
        if (threadIdx.x == 0) cnt[t] = s_c;
    } else {
        uint32_t tot;
        uint32_t o = off[t] + block_excl_scan((uint32_t)__popc(flags), s_scan, tot);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (flags & (1u << j)) out[o++] = v[j];
    }
}

// Per pending cell: its resident position, or kChgNone when it is below min_points.  keys = D (n = *n_ptr entries), or null
// for "every resident cell" (n = *n_ptr resident cells, position = index).  A key of D that is not resident raises *err.
// cnt[t] = the tile's emitted cells.
__global__ void __launch_bounds__(kThreads) k_chg_emit_cnt(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ n_ptr,
                                                           const uint64_t* __restrict__ res_keys,
                                                           const uint32_t* __restrict__ n_res_ptr,
                                                           const float4* __restrict__ res_acc, uint32_t min_points,
                                                           uint32_t* __restrict__ pos, uint32_t* __restrict__ cnt,
                                                           uint32_t* __restrict__ err) {
    wait_prior();
    const uint32_t n = *n_ptr, n_res = *n_res_ptr;
    const uint32_t t = blockIdx.x;
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t i = t * kTileV + threadIdx.x * 4 + j;
        if (i >= n) continue;
        uint32_t p = i;
        if (keys) {
            const uint64_t k = keys[i];
            uint32_t lo = 0, hi = n_res;   // lower_bound in the resident keys
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (res_keys[mid] < k) lo = mid + 1; else hi = mid;
            }
            if (lo >= n_res || res_keys[lo] != k) { atomicOr(err, 1u); lo = kChgNone; }
            p = lo;
        }
        if (p != kChgNone && __float_as_uint(res_acc[p].w) < min_points) p = kChgNone;
        pos[i] = p;
        if (p != kChgNone) ++c;
    }
    c = __reduce_add_sync(kFull, c);
    __shared__ uint32_t s_c;
    if (threadIdx.x == 0) s_c = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_c, c);
    __syncthreads();
    if (threadIdx.x == 0) cnt[t] = s_c;
}

// the records of the cells k_chg_emit_cnt selected, in D's (= key) order: point (acc_centroid), key, point count
__global__ void __launch_bounds__(kThreads) k_chg_emit(const uint32_t* __restrict__ n_ptr, const uint32_t* __restrict__ pos,
                                                       const uint64_t* __restrict__ res_keys, const float4* __restrict__ res_acc,
                                                       const uint4* __restrict__ res_rgb, const uint32_t* __restrict__ off,
                                                       float4* __restrict__ out, uint64_t* __restrict__ out_keys,
                                                       uint32_t* __restrict__ out_counts) {
    wait_prior();
    __shared__ uint32_t s_scan[34];
    const uint32_t n = *n_ptr;
    const uint32_t t = blockIdx.x;
    uint32_t p[4], flags = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t i = t * kTileV + threadIdx.x * 4 + j;
        p[j] = i < n ? pos[i] : kChgNone;
        if (p[j] != kChgNone) flags |= 1u << j;
    }
    uint32_t tot;
    uint32_t o = off[t] + block_excl_scan((uint32_t)__popc(flags), s_scan, tot);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (!(flags & (1u << j))) continue;
        const float4 a = res_acc[p[j]];
        out[o] = acc_centroid(a, res_rgb[p[j]]);
        out_keys[o] = res_keys[p[j]];
        out_counts[o] = __float_as_uint(a.w);
        ++o;
    }
}

}  // namespace o3r
