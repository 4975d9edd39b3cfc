// prereduce.cuh — tile-local pre-reduction of the cycle's per-frame voxel centroids on the combined grid
// (O3R_MERGE_ACCUMULATE_TILED).
//
// downsamplePtCloud(cloud_big, true) (pose_functions.cpp:1654-1709) sums, per (voxel_size, voxel_size, 1000) cell, every
// point that was ever appended to cloud_big.  The exact-order engine (voxel.cuh, engine 2) sorts all of a cycle's
// items by cell and left-folds them; that moves ~150 B per item.  Here a CTA takes 1024 CONSECUTIVE items of the
// per-frame voxel list (sorted by the fine (k, j, i) index, so a tile touches ~120 combined cells), groups them by
// cell inside shared memory and emits one partial sum per distinct cell: 8x fewer records reach the sort + merge.
//
// Grouping: open-addressing hash of the 64-bit cell key (atomicCAS) -> dense bin ids (scan over the table) ->
// stable counting sort of the tile by bin id (warp match_any ranks + warp-private counters, as in the radix pass)
// -> one thread per bin left-folds its items in tile order.  Which table slot a key lands in depends on a race, but
// only the order of DIFFERENT cells' records inside the tile's output depends on that; every partial is a fixed
// left fold of fixed items, tiles write in ticket order at offsets from a decoupled look-back, and the sort after this
// is stable, so the final sums are reproducible bit for bit from run to run.  They differ from the oracle's single
// left fold over all points by float reassociation only (keys, counts and colour sums are exact).
#pragma once
#include "common.cuh"
#include "sort.cuh"

namespace o3r {

constexpr int kPrItems = 4;
constexpr int kPrTile = kThreads * kPrItems;     // 1024 items per CTA
constexpr int kPrTab = 2 * kPrTile;              // hash table entries (load <= 0.5)
constexpr unsigned long long kPrEmpty = ~0ull;   // absolute cell keys use 63 bits

struct PrSmem {
    union {
        struct { unsigned long long tab[kPrTab]; uint16_t dense[kPrTab]; } h;   // grouping phase
        float4 items[kPrTile];                                                  // tile in bin order (sum phase)
    } u;
    uint16_t cnt[kWarps][kPrTile];   // per warp and bin: count, then exclusive prefix over the warps
    uint16_t base[kPrTile + 1];      // bin b occupies items[base[b], base[b + 1])
    uint16_t tot[kPrTile];           // items per bin
    uint32_t scan[34];
    uint32_t ticket, out0, nb;
};

// in:  items [*in_base, *in_base + *in_count) of `vox` (per-frame voxel centroids of the chunk, {x, y, z, 0x00RRGGBB})
// out: partial cells appended at out[*out_base ...); *chunk_total receives how many (k_add_u32 then advances the base)
// status/ticket: zeroed by the caller; one status word per tile (flag << 30 | count).
__global__ void __launch_bounds__(kThreads, 5) k_cell_prereduce(const float4* __restrict__ vox,
                                                                const uint32_t* __restrict__ in_base,
                                                                const uint32_t* __restrict__ in_count, float icx, float icz,
                                                                o3r_cell* __restrict__ out,
                                                                const uint32_t* __restrict__ out_base,
                                                                uint32_t* __restrict__ chunk_total,
                                                                uint32_t* __restrict__ status, uint32_t* __restrict__ ticket) {
    wait_prior();
    __shared__ PrSmem S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    if (tid == 0) { S.ticket = atomicAdd(ticket, 1u); S.nb = 0; }
    const uint32_t n = *in_count, ibase = *in_base, obase = *out_base;
    // ---- clear the table (128-bit stores)
    {
        uint4* tz = reinterpret_cast<uint4*>(S.u.h.tab);
#pragma unroll
        for (int i = 0; i < kPrTab / 2 / kThreads; ++i) tz[i * kThreads + tid] = make_uint4(~0u, ~0u, ~0u, ~0u);
    }
    __syncthreads();
    const uint32_t t = S.ticket;
    if (t * kPrTile >= n) return;
    const uint32_t nt = (n + kPrTile - 1) / kPrTile;
    const uint32_t wn = min((uint32_t)kPrTile, n - t * kPrTile);
    vox += ibase + t * kPrTile;
    // ---- load: warp w owns items [w*128, w*128 + 128) as 4 rounds of 32 consecutive items
    float4 it[kPrItems];
    unsigned long long key[kPrItems];
    uint32_t slot[kPrItems];
#pragma unroll
    for (int r = 0; r < kPrItems; ++r) {
        const uint32_t e = warp * (32 * kPrItems) + r * 32 + lane;
        key[r] = kPrEmpty;
        if (e < wn) {
            it[r] = __ldcs(vox + e);
            it[r].z = __fadd_rn(it[r].z, 500.0f);   // pose_functions.cpp:1666
            key[r] = abs_cell_key(it[r].x, it[r].y, it[r].z, icx, icx, icz);
        }
    }
    // ---- one table slot per distinct cell; whoever creates the slot numbers the bin
#pragma unroll
    for (int r = 0; r < kPrItems; ++r) {
        slot[r] = 0;
        if (key[r] != kPrEmpty) {
            unsigned long long k = key[r];
            uint32_t h = (uint32_t)(k ^ (k >> 21) ^ (k >> 42)) * 0x9e3779b1u;
            h >>= 32 - 11;   // kPrTab = 2048
            for (;;) {
                const unsigned long long old = atomicCAS(&S.u.h.tab[h], kPrEmpty, k);
                if (old == kPrEmpty) { S.u.h.dense[h] = (uint16_t)atomicAdd(&S.nb, 1u); break; }
                if (old == k) break;
                h = (h + 1) & (kPrTab - 1);
            }
            slot[r] = h;
        }
    }
    __syncthreads();
    const uint32_t nb = S.nb;
    // publish the tile's record count early: the successors' look-back rarely has to wait
    if (tid == 0) st_volatile_u32(status + t, (t == 0 ? kStGlobal : kStLocal) | nb);
    // the counters of the live bins (and of the stand-in bin of lanes without an item)
    for (uint32_t b = tid; b < nb; b += kThreads) {
#pragma unroll
        for (int w = 0; w < kWarps; ++w) S.cnt[w][b] = 0;
    }
    if (tid < kWarps) S.cnt[tid][kPrTile - 1] = 0;
    __syncthreads();
    // ---- stable rank of every item inside its bin (tile order = warp, round, lane)
    // lanes without an item use bin kPrTile-1, which no real bin can be unless the tile is full (nb <= wn)
    uint32_t bin[kPrItems], rk[kPrItems];
    uint16_t* wc = &S.cnt[warp][0];
#pragma unroll
    for (int r = 0; r < kPrItems; ++r) {
        const bool valid = key[r] != kPrEmpty;
        bin[r] = valid ? (uint32_t)S.u.h.dense[slot[r]] : (uint32_t)(kPrTile - 1);
        const unsigned peers = __match_any_sync(kFull, valid ? bin[r] : 0xffffffffu);
        const uint32_t old = wc[bin[r]];
        __syncwarp();
        if (valid && (peers & lt) == 0u) wc[bin[r]] = (uint16_t)(old + __popc(peers));
        __syncwarp();
        rk[r] = old + __popc(peers & lt);
    }
    __syncthreads();
    // ---- per bin: exclusive prefix over the warps, then the bins' start positions
    for (uint32_t b = tid; b < nb; b += kThreads) {
        uint32_t c[kWarps], acc = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) c[w] = S.cnt[w][b];
#pragma unroll
        for (int w = 0; w < kWarps; ++w) { S.cnt[w][b] = (uint16_t)acc; acc += c[w]; }
        S.tot[b] = (uint16_t)acc;
    }
    __syncthreads();
    {
        uint32_t run[kPrItems], rsum = 0;
#pragma unroll
        for (int q = 0; q < kPrItems; ++q) {
            const uint32_t b = tid * kPrItems + q;
            run[q] = b < nb ? (uint32_t)S.tot[b] : 0u;
            rsum += run[q];
        }
        uint32_t tot;
        uint32_t ds = block_excl_scan(rsum, S.scan, tot);
#pragma unroll
        for (int q = 0; q < kPrItems; ++q) { S.base[tid * kPrItems + q] = (uint16_t)ds; ds += run[q]; }
        if (tid == kThreads - 1) S.base[kPrTile] = (uint16_t)tot;
    }
    __syncthreads();   // (the table is dead from here on: `items` aliases it)
#pragma unroll
    for (int r = 0; r < kPrItems; ++r)
        if (key[r] != kPrEmpty) S.u.items[(uint32_t)S.base[bin[r]] + (uint32_t)wc[bin[r]] + rk[r]] = it[r];
    // ---- where the tile's records go: decoupled look-back over the predecessors' counts, 32 tiles per step
    // (the tiles of a wave reach this point together, so most predecessors are still LOCAL: a one-thread walk
    // would cross hundreds of them one L2 round trip at a time)
    if (warp == 0) {
        uint32_t pf = 0;
        for (int32_t back = (int32_t)t - 1; back >= 0; back -= 32) {
            const int32_t idx = back - lane;
            uint32_t v = kStGlobal;   // before tile 0: an inclusive prefix of 0
            if (idx >= 0)
                while (((v = ld_volatile_u32(status + idx)) >> 30) == 0u) __nanosleep(32);
            const unsigned gm = __ballot_sync(kFull, (v >> 30) == 2u);
            const int first = gm ? __ffs(gm) - 1 : 31;
            pf += __reduce_add_sync(kFull, lane <= first ? (v & kStMask) : 0u);
            if (gm) break;
        }
        if (lane == 0) {
            if (t > 0) st_volatile_u32(status + t, kStGlobal | (pf + nb));
            S.out0 = pf;
            if (t == nt - 1) *chunk_total = pf + nb;
        }
    }
    __syncthreads();
    out += obase + S.out0;
    // ---- one thread per bin: left fold in tile order
    for (uint32_t b = tid; b < nb; b += kThreads) {
        const uint32_t a = S.base[b], e = S.base[b + 1];
        const float4 p0 = S.u.items[a];
        float sx = 0.f, sy = 0.f, sz = 0.f;
        uint32_t cr = 0, cg = 0, cb = 0;
        for (uint32_t i = a; i < e; ++i) {
            const float4 p = S.u.items[i];
            sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z);
            const uint32_t w = __float_as_uint(p.w);
            cr += (w >> 16) & 255u; cg += (w >> 8) & 255u; cb += w & 255u;
        }
        o3r_cell c;
        c.key = abs_cell_key(p0.x, p0.y, p0.z, icx, icx, icz);
        c.sx = sx; c.sy = sy; c.sz = sz; c.n = e - a;
        c.sr = cr; c.sg = cg; c.sb = cb; c.pad = 0;
        out[b] = c;
    }
}

__global__ void k_add_u32(uint32_t* dst, const uint32_t* src) {
    wait_prior();
    if (threadIdx.x == 0) *dst += *src;
}

}  // namespace o3r
