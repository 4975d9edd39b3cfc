// retain.cuh — device side of the sharded RETAIN downsample (host_retain.cuh): the retained cloud stays where its frames were
// reconstructed, and o3r_cloud_downsample moves every point once to the rank that owns its combined-grid cell.  The owner then
// restores the single-GPU order of its points (cloud_big order: cycle, frame, index in frame) from a per-point order tag and
// runs engine 1 (voxel.cuh) on them with the global grid, so its centroids are the single-GPU ones bit for bit.
#pragma once
#include "common.cuh"
#include "sort.cuh"
#include "voxel.cuh"

namespace o3r {

// one point on its way to its owner: the point as stored (x, y, z, packed colour) and its order tag
struct RtRec { float x, y, z; uint32_t rgb, tag; };   // 20 bytes
// one appended frame of the local cloud: its first point, its cycle and its global frame index (order tag: cycle << frame bits
// | frame, with the frame bits agreed at each downsample)
struct RtFrameDev { uint32_t first, cycle, frame; };

// Points a rank may hold or own: 32-bit indices, and a margin of 2^24 keeps every grid-stride loop of the path (at most
// 148 * 16 CTAs of 256 threads per stride) and its warp-rounded bound clear of 2^32.
constexpr size_t kRtMaxPoints = (1ull << 32) - (1ull << 24);
constexpr int kRtWords = 16;   // words of the first agreement (all-reduced with max)
enum { RT_W_BBOX = 0, RT_W_FRAMES = 6, RT_W_CYCLES = 7, RT_W_ERR = 8, RT_W_WRAP = 9 };

// the local z-shifted bbox (k_bbox_pts) and the rank's frame / cycle ranges -> the words the ranks combine with max: the
// minimum corner travels complemented, so one max-reduction yields min and max of the order-preserving encoding
__global__ void k_rt_agree_pack(const uint32_t* __restrict__ bbox, uint32_t n_frames, uint32_t n_cycles, uint32_t err,
                                uint32_t* __restrict__ w) {
    wait_prior();
    const int t = threadIdx.x;
    if (t < 3) w[RT_W_BBOX + t] = ~bbox[t];
    else if (t < 6) w[RT_W_BBOX + t] = bbox[t];
    else if (t == RT_W_FRAMES) w[t] = n_frames;
    else if (t == RT_W_CYCLES) w[t] = n_cycles;
    else if (t == RT_W_ERR) w[t] = err;
    else if (t < kRtWords) w[t] = 0u;
}

// the combined words -> the global bbox and PCL's grid (every rank computes identical GridParams, pass-through verdict
// included).  RT_W_WRAP flags a grid of more than 2^32 cells: there PCL's wrapped 32-bit index can merge distinct absolute
// cells, which the owner hash would keep apart.
__global__ void k_rt_grid(uint32_t* __restrict__ w, float ix, float iy, float iz, uint32_t* __restrict__ bbox,
                          GridParams* __restrict__ grid) {
    wait_prior();
    if (threadIdx.x != 0) return;
    uint32_t bb[6];
    for (int a = 0; a < 3; ++a) { bb[a] = ~w[RT_W_BBOX + a]; bb[3 + a] = w[RT_W_BBOX + 3 + a]; }
    for (int a = 0; a < 6; ++a) bbox[a] = bb[a];
    const GridParams G = make_grid(bb, ix, iy, iz);
    *grid = G;
    uint32_t wrap = 0;
    if (!G.empty && !G.passthrough) {
        const float inv[3] = {ix, iy, iz};
        unsigned long long cells = 1;
        for (int a = 0; a < 3; ++a)
            cells *= (unsigned long long)((int)floorf(__fmul_rn(ord2f(bb[3 + a]), inv[a])) - G.min_b[a] + 1);
        wrap = cells > (1ull << 32);
    }
    w[RT_W_WRAP] = wrap;
}

// per local point: owner rank of its combined-grid cell (keys), order tag (tags), per-owner histogram (counts, pass 0 of
// the one-pass owner sort).  The frame of point i is the last table entry whose first point is <= i.
__global__ void __launch_bounds__(kThreads) k_rt_route(const float4* __restrict__ pts, uint32_t n, const RtFrameDev* __restrict__ ftab,
                                                       uint32_t n_frames, uint32_t fbits, float ix, float iy, float iz, uint32_t world,
                                                       uint32_t* __restrict__ okeys, uint32_t* __restrict__ tags,
                                                       uint32_t* __restrict__ counts) {
    wait_prior();
    __shared__ uint32_t s_cnt[256];   // (world <= 256)
    for (uint32_t r = threadIdx.x; r < world; r += kThreads) s_cnt[r] = 0u;
    __syncthreads();
    const uint32_t n_round = (n + 31u) & ~31u;   // whole warps take every trip (match_any below)
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n_round; i += gridDim.x * kThreads) {
        uint32_t o = 0xffffffffu;
        if (i < n) {
            const float4 p = pts[i];
            o = (uint32_t)(hash64(abs_cell_key(p.x, p.y, __fadd_rn(p.z, 500.0f), ix, iy, iz)) % world);
            uint32_t lo = 0, hi = n_frames;   // invariant: ftab[lo].first <= i (entry 0 starts at point 0)
            while (hi - lo > 1) {
                const uint32_t mid = (lo + hi) >> 1;
                if (ftab[mid].first <= i) lo = mid; else hi = mid;
            }
            okeys[i] = o;
            tags[i] = (ftab[lo].cycle << fbits) | ftab[lo].frame;
        }
        const unsigned peers = __match_any_sync(kFull, o);
        if (o != 0xffffffffu && (peers & ((1u << (threadIdx.x & 31)) - 1u)) == 0u) atomicAdd(&s_cnt[o], (uint32_t)__popc(peers));
    }
    __syncthreads();
    for (uint32_t r = threadIdx.x; r < world; r += kThreads)
        if (s_cnt[r]) atomicAdd(&counts[r], s_cnt[r]);
}

// points in owner order (perm = the stable owner sort's values) -> the send buffer, one contiguous bucket per owner
__global__ void __launch_bounds__(kThreads) k_rt_pack(const float4* __restrict__ pts, const uint32_t* __restrict__ tags,
                                                      const uint32_t* __restrict__ perm, uint32_t n, RtRec* __restrict__ out) {
    wait_prior();
    for (uint32_t j = blockIdx.x * kThreads + threadIdx.x; j < n; j += gridDim.x * kThreads) {
        const uint32_t i = perm[j];
        const float4 p = pts[i];
        RtRec r;
        r.x = p.x; r.y = p.y; r.z = p.z; r.rgb = __float_as_uint(p.w); r.tag = tags[i];
        out[j] = r;
    }
}

// per-destination counts + a clear status word: the counts agreement of a rank whose routing succeeded (a failed rank
// writes zero counts and a set status from the host instead)
__global__ void k_rt_counts(const uint32_t* __restrict__ counts, uint32_t world, uint32_t* __restrict__ out) {
    wait_prior();
    for (uint32_t d = threadIdx.x; d < world; d += blockDim.x) {
        out[2 * d] = counts[d];
        out[2 * d + 1] = 0u;
    }
}

__global__ void __launch_bounds__(kThreads) k_rt_tags(const RtRec* __restrict__ rec, uint32_t n, uint32_t* __restrict__ keys) {
    wait_prior();
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) keys[i] = rec[i].tag;
}

// received records in tag order (the stable tag sort's values; identity when no pass ran) -> points in cloud_big order
__global__ void __launch_bounds__(kThreads) k_rt_gather(const RtRec* __restrict__ rec, uint32_t n, const SortPlan* __restrict__ plan,
                                                        const uint32_t* __restrict__ v0, const uint32_t* __restrict__ v1,
                                                        float4* __restrict__ out) {
    wait_prior();
    const bool ident = plan->n_active == 0;
    const uint32_t* perm = plan->final_parity ? v1 : v0;
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        const RtRec r = rec[ident ? i : perm[i]];
        out[i] = make_float4(r.x, r.y, r.z, __uint_as_float(r.rgb));
    }
}

}  // namespace o3r
