// sort.cuh — hand-written segmented LSD radix sort of (key, u32 value) pairs, plus the exclusive-scan
// kernel the pipeline uses.  No Thrust / CUB.
//
// Digits are up to kRsMaxBits wide and sized per segment: k_rs_layout splits the segment's live key bits evenly
// over the fewest passes (28-bit per-frame voxel index -> 7+7+7+7, 20-bit combined-grid key -> 7+7+6).
// k_rs_ghist reads the keys once and builds every pass's whole-segment digit histogram; each pass is then
// ONE kernel (k_rs_onesweep): stable in-tile ranking with warp match_any, tile offsets by decoupled
// look-back, exchange through shared memory so that every digit run leaves the CTA as one coalesced burst.
// Stability is what makes the later per-voxel sums run in input order (bit-exact with the oracle's stable
// order).
//
// Segments (one per frame for the per-frame grid, a single one for the combined grid) are described
// by a device array seg_off[S+1]; launches are sized by a host upper bound and surplus CTAs exit.
// The per-segment SortPlan also skips passes whose digit is constant over the segment and whole
// segments that need no sorting (PCL pass-through frames).
#pragma once
#include "common.cuh"

namespace o3r {

#ifndef O3R_RS_ITEMS
#define O3R_RS_ITEMS 16
#endif
#ifndef O3R_RS_MINB
#define O3R_RS_MINB 4
#endif
// In-warp peer search of the ranking loop: 0 = match.any, 1 = shared-memory atomicOr on a per-warp mask per digit.
#ifndef O3R_RS_RANK
#define O3R_RS_RANK 1
#endif
constexpr int kRsItems = O3R_RS_ITEMS;
constexpr int kRsTile = kThreads * kRsItems;  // 4096 pairs per CTA
// Measured on B200 (r01): 10-bit digits save a pass (28-bit index: 3 instead of 4) but the per-tile bin work
// (warps x bins counters to prefix, 4 look-backs per thread) makes each pass ~50 % slower; 8 bits wins.
#ifndef O3R_RS_BITS
#define O3R_RS_BITS 8
#endif
constexpr int kRsMaxBits = O3R_RS_BITS;
constexpr int kRsBins = 1 << kRsMaxBits;      // bins at most per pass
constexpr int kRsBpt = kRsBins / kThreads;    // bins per thread
constexpr int kMaxPasses = 8;

struct SortPlan {
    uint32_t active_mask;    // bit p: pass p runs
    uint32_t parity_mask;    // bit p: pass p reads ping-pong buffer 1
    uint32_t final_parity;   // buffer holding the sorted result
    uint32_t n_active;
    uint32_t n_passes;
    uint8_t shift[kMaxPasses];
    uint8_t bits[kMaxPasses];
};

// ---- generic single-segment exclusive scan (one CTA of 1024 threads, 4 per thread and iteration, carry across iterations) ----
// The inputs are per-tile counts (tens of thousands of words): one wide CTA finishes them in a handful of iterations.
constexpr int kScanThreads = 1024;
__global__ void __launch_bounds__(kScanThreads) k_scan_u32(const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                           uint32_t n, uint32_t* __restrict__ total_out) {
    __shared__ uint32_t s_w[32];
    __shared__ uint32_t s_tot;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t carry = 0;
    for (uint32_t base = 0; base < n; base += kScanThreads * 4) {
        const uint32_t i = base + threadIdx.x * 4;
        uint32_t v[4];
        if (i + 3 < n && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
            const uint4 q = *reinterpret_cast<const uint4*>(in + i);
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = (i + j < n) ? in[i + j] : 0u;
        }
        const uint32_t mine = v[0] + v[1] + v[2] + v[3];
        uint32_t inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) s_w[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            const uint32_t w = s_w[lane];
            uint32_t winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(kFull, winc, o);
                if (lane >= o) winc += t;
            }
            s_w[lane] = winc - w;
            if (lane == 31) s_tot = winc;
        }
        __syncthreads();
        uint32_t off = carry + s_w[warp] + inc - mine;
        const uint32_t tot = s_tot;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (i + j < n) out[i + j] = off;
            off += v[j];
        }
        carry += tot;
    }
    if (threadIdx.x == 0 && total_out) *total_out = carry;
}

// ---- digit layout: split `key_bits` live bits into the fewest passes of <= 10 bits -------------------------------
// key_bits comes from the segment's VoxelGrid (grids[s].key_bits) or is the same for all segments (fixed_bits).
__global__ void k_rs_layout(int n_seg, const GridParams* __restrict__ grids, int fixed_bits, SortPlan* __restrict__ plan) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    int kb = grids ? grids[s].key_bits : fixed_bits;
    kb = max(1, min(kb, 64));
    const int np = (kb + kRsMaxBits - 1) / kRsMaxBits;
    const int base = kb / np, rem = kb - base * np;
    SortPlan pl;
    pl.active_mask = pl.parity_mask = pl.final_parity = pl.n_active = 0;
    pl.n_passes = np;
    int sh = 0;
    for (int p = 0; p < kMaxPasses; ++p) {
        const int w = p < np ? base + (p < rem ? 1 : 0) : 0;
        pl.shift[p] = (uint8_t)sh;
        pl.bits[p] = (uint8_t)w;
        sh += w;
    }
    plan[s] = pl;
}

// ---- which passes run: skip digits that are constant over the segment and segments that need no sorting ---------
// ghist[S][kMaxPasses][kRsBins]
// Finally turns each pass's histogram into its exclusive prefix (where every digit's run starts in the segment), which
// is what the radix pass needs: computed once here instead of once per tile.
__global__ void __launch_bounds__(kThreads) k_rs_plan(uint32_t* __restrict__ ghist, const uint32_t* __restrict__ seg_off,
                                                      SortPlan* __restrict__ plan, const GridParams* __restrict__ grids) {
    __shared__ int s_trivial[kMaxPasses];
    __shared__ uint32_t s_scan[34];
    const int s = blockIdx.x;
    const uint32_t n = seg_off[s + 1] - seg_off[s];
    const int np = plan[s].n_passes;
    if (threadIdx.x < kMaxPasses) s_trivial[threadIdx.x] = 0;
    __syncthreads();
    for (int p = 0; p < np; ++p)
        for (int b = threadIdx.x; b < kRsBins; b += kThreads)
            if (ghist[((size_t)s * kMaxPasses + p) * kRsBins + b] == n) s_trivial[p] = 1;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t am = 0, pm = 0, par = 0, na = 0;
        for (int p = 0; p < kMaxPasses; ++p) {
            const bool act = p < np && n > 0 && !s_trivial[p] && !(grids && grids[s].passthrough);
            if (act) am |= 1u << p;
            if (par) pm |= 1u << p;
            if (act) { par ^= 1u; ++na; }
        }
        plan[s].active_mask = am;
        plan[s].parity_mask = pm;
        plan[s].final_parity = par;
        plan[s].n_active = na;
    }
    for (int p = 0; p < np; ++p) {
        uint32_t* gh = ghist + ((size_t)s * kMaxPasses + p) * kRsBins + threadIdx.x * kRsBpt;
        uint32_t h[kRsBpt], sum = 0;
#pragma unroll
        for (int q = 0; q < kRsBpt; ++q) { h[q] = gh[q]; sum += h[q]; }
        uint32_t tot;
        uint32_t e = block_excl_scan(sum, s_scan, tot);
#pragma unroll
        for (int q = 0; q < kRsBpt; ++q) { gh[q] = e; e += h[q]; }
    }
}

template <typename KeyT>
__device__ __forceinline__ uint32_t rs_digit(KeyT k, int shift, uint32_t mask) { return (uint32_t)(k >> shift) & mask; }

// shared-memory histogram update by the lanes of `vm`: one aggregated atomic when the whole warp agrees on the
// digit (the constant high digits that would otherwise serialise), plain atomics otherwise
__device__ __forceinline__ void hist_add(uint32_t* sh, uint32_t d, unsigned vm, int lane) {
    int uniform;
    __match_all_sync(vm, d, &uniform);
    if (uniform) {
        if (lane == __ffs(vm) - 1) atomicAdd(&sh[d], (uint32_t)__popc(vm));
    } else {
        atomicAdd(&sh[d], 1u);
    }
}

// ---- whole-segment digit histograms for every pass in one read of the keys ------------------------------------
// ghist[S][kMaxPasses][kRsBins]; must be zeroed by the caller.  MAXP bounds the passes of this key type.
template <typename KeyT, int MAXP>
__global__ void __launch_bounds__(kThreads) k_rs_ghist(const KeyT* __restrict__ keys, const uint32_t* __restrict__ seg_off,
                                                       const SortPlan* __restrict__ plan, uint32_t* __restrict__ ghist) {
    __shared__ uint32_t sh[MAXP * kRsBins];
    const int s = blockIdx.y;
    const uint32_t t = blockIdx.x;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    if (t * kRsTile >= n) return;
    const int np = min((int)plan[s].n_passes, MAXP);
    int shift[MAXP];
    uint32_t mask[MAXP];
#pragma unroll
    for (int p = 0; p < MAXP; ++p) { shift[p] = plan[s].shift[p]; mask[p] = (1u << plan[s].bits[p]) - 1u; }
    for (int i = threadIdx.x; i < MAXP * kRsBins; i += kThreads) sh[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll 2
    for (int r = 0; r < kRsItems; ++r) {
        const uint32_t i = t * kRsTile + warp * (32 * kRsItems) + r * 32 + lane;
        const bool valid = i < n;
        const unsigned vm = __ballot_sync(kFull, valid);
        if (valid) {
            const KeyT k = keys[beg + i];
#pragma unroll
            for (int p = 0; p < MAXP; ++p)
                if (p < np) hist_add(sh + p * kRsBins, rs_digit(k, shift[p], mask[p]), vm, lane);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < MAXP * kRsBins; i += kThreads)
        if (sh[i]) atomicAdd(&ghist[(size_t)s * kMaxPasses * kRsBins + i], sh[i]);
}

// ---- one radix pass in one kernel: stable in-tile rank, decoupled look-back for the tile's digit offsets ---------
// ("onesweep"): every tile publishes its per-digit counts in status[seg][tile][1024] (2 flag bits + 30 count
// bits in one word), then each thread walks back over the predecessors' words of ITS digit(s) until it
// meets an inclusive prefix.  A digit's inclusive prefix counts up to the whole segment: segments that can reach
// 2^30 items use the 64-bit status word instead (StT = uint64_t: 2 flag bits + 62 count bits).  Tiles take their index from an atomic ticket so a predecessor is always resident
// or finished before anyone waits on it.
// Dynamic shared memory: pairs[4096] (key, value) | cnt[kWarps][bins] u16 | gbase[bins] u32 | scan
template <typename KeyT>
struct RsPair { KeyT k; uint32_t v; };
template <>
struct __align__(8) RsPair<uint32_t> { uint32_t k; uint32_t v; };

template <typename KeyT>
constexpr size_t rs_scatter_smem() {
    return (size_t)kRsTile * sizeof(RsPair<KeyT>) + (size_t)kWarps * kRsBins * 2 + (size_t)kRsBins * 4 + 36 * 4 +
           (O3R_RS_RANK == 1 && sizeof(KeyT) == 4 ? (size_t)kWarps * kRsBins * 4 : 0);
}

constexpr uint32_t kStLocal = 1u << 30, kStGlobal = 2u << 30, kStMask = (1u << 30) - 1u;
// segments of at least this many items sort with 64-bit look-back words
constexpr size_t kRsWideSeg = (size_t)1 << 30;

// flag + payload live in ONE word, so relaxed gpu-scope accesses are enough (no fence, no system scope)
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_status(const uint32_t* p) { return ld_volatile_u32(p); }
__device__ __forceinline__ void st_status(uint32_t* p, uint32_t v) { st_volatile_u32(p, v); }
__device__ __forceinline__ uint64_t ld_status(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_status(uint64_t* p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

template <typename KeyT, typename StT>
__global__ void __launch_bounds__(kThreads, sizeof(KeyT) == 4 ? O3R_RS_MINB : (O3R_RS_MINB > 3 ? 3 : O3R_RS_MINB)) k_rs_onesweep(
    KeyT* __restrict__ keys0, KeyT* __restrict__ keys1, uint32_t* __restrict__ vals0, uint32_t* __restrict__ vals1,
    const uint32_t* __restrict__ seg_off, const SortPlan* __restrict__ plan, int pass, uint32_t tiles_ub,
    const uint32_t* __restrict__ ghist, StT* __restrict__ status, uint32_t* __restrict__ ticket, int iota_first,
    int ghist_is_prefix) {
    constexpr int kFlagShift = (int)sizeof(StT) * 8 - 2;
    constexpr StT kLocal = (StT)1 << kFlagShift, kGlobal = (StT)2 << kFlagShift, kCountMask = kLocal - 1;
    extern __shared__ __align__(16) unsigned char rs_smem[];
    RsPair<KeyT>* s_pairs = reinterpret_cast<RsPair<KeyT>*>(rs_smem);
    uint16_t* cnt = reinterpret_cast<uint16_t*>(rs_smem + (size_t)kRsTile * sizeof(RsPair<KeyT>));   // [kWarps][1024]
    uint32_t* gbase = reinterpret_cast<uint32_t*>(cnt + kWarps * kRsBins);   // [1024] destination of local position i: gbase[d] + i
    uint32_t* s_scan = gbase + kRsBins;                                      // [34]
    uint32_t* s_ticket = s_scan + 34;
    // 32-bit keys only: with 16-byte pairs the extra 8 KB would cost the third resident CTA
    constexpr bool kOrMask = O3R_RS_RANK == 1 && sizeof(KeyT) == 4;
    uint32_t* wmask = s_ticket + 2;                                          // [kWarps][kRsBins] lanes holding digit d (kOrMask)

    if (threadIdx.x == 0) *s_ticket = atomicAdd(ticket, 1u);
    __syncthreads();
    // Tickets go round-robin over the segments (tile 0 of every segment, then tile 1 of every segment, ...): the CTAs
    // resident at any moment are then a few consecutive tiles of EACH segment, and a tile's look-back meets an inclusive
    // prefix after a handful of predecessors.  Segment-major tickets put all ~180 tiles of a frame in flight together,
    // every one of them still LOCAL, and each look-back walked back to tile 0 (O(tiles^2) status reads per segment).
    const uint32_t lin = *s_ticket;
    const uint32_t n_seg = gridDim.x / tiles_ub;
    const int s = (int)(lin % n_seg);
    const uint32_t t = lin / n_seg;
    const uint32_t amask = plan[s].active_mask;
    if (!((amask >> pass) & 1u)) return;
    const uint32_t beg = seg_off[s], n = seg_off[s + 1] - beg;
    const uint32_t nt = (n + kRsTile - 1) / kRsTile;
    if (t >= nt) return;

    const int par = (plan[s].parity_mask >> pass) & 1u;
    const int shift = plan[s].shift[pass];
    const uint32_t nb = 1u << plan[s].bits[pass], dmask = nb - 1u;
    const KeyT* kin = (par ? keys1 : keys0) + beg;
    const uint32_t* vin = (par ? vals1 : vals0) + beg;
    KeyT* kout = (par ? keys0 : keys1) + beg;
    uint32_t* vout = (par ? vals0 : vals1) + beg;
    const bool first = (amask & ((1u << pass) - 1u)) == 0u;   // no active pass before this one
    const bool iota = iota_first && first;   // values are the global element index, not read from memory
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int b0 = threadIdx.x * kRsBpt;   // this thread's bin(s)

    {   // every warp zeroes ITS OWN u16 counters (no CTA barrier stands between this and the ranking loop)
        uint32_t* cz = reinterpret_cast<uint32_t*>(cnt + warp * kRsBins);
#pragma unroll
        for (int i = 0; i < kRsBins / 2 / 32; ++i) cz[i * 32 + lane] = 0u;
        if constexpr (kOrMask) {
#pragma unroll
            for (int i = 0; i < kRsBins / 32; ++i) wmask[warp * kRsBins + i * 32 + lane] = 0u;
        }
        __syncwarp();
    }
    // exclusive scan of the segment's digit histogram = where each digit's run starts in the segment
    uint32_t dbase[kRsBpt];
    {
        const uint32_t* gh = ghist + ((size_t)s * kMaxPasses + pass) * kRsBins + b0;
        if (ghist_is_prefix) {   // k_rs_plan already scanned it
#pragma unroll
            for (int q = 0; q < kRsBpt; ++q) dbase[q] = gh[q];
        } else {
            uint32_t h[kRsBpt], sum = 0;
#pragma unroll
            for (int q = 0; q < kRsBpt; ++q) { h[q] = gh[q]; sum += h[q]; }
            uint32_t tot;
            uint32_t e = block_excl_scan(sum, s_scan, tot);
#pragma unroll
            for (int q = 0; q < kRsBpt; ++q) { dbase[q] = e; e += h[q]; }
        }
    }

    KeyT key[kRsItems];
    uint32_t rk[kRsItems / 2];   // two 16-bit in-warp ranks per word
    const uint32_t wbase = t * kRsTile + warp * (32 * kRsItems);
    const uint32_t ntile = min((uint32_t)kRsTile, n - t * kRsTile);
    const bool full = ntile == (uint32_t)kRsTile;   // no bounds checks in a full tile
    {
        const KeyT* kp = kin + wbase + lane;
        if (full) {
#pragma unroll
            for (int r = 0; r < kRsItems; ++r) key[r] = kp[r * 32];
        } else {
#pragma unroll
            for (int r = 0; r < kRsItems; ++r) key[r] = (wbase + r * 32 + lane < n) ? kp[r * 32] : ~(KeyT)0;
        }
    }
    uint16_t* wc = cnt + warp * kRsBins;
    uint32_t* wm = wmask + warp * kRsBins;
#pragma unroll
    for (int r = 0; r < kRsItems; ++r) {
        // padding items carry the highest digit and sit at the very end of the tile order, so they never
        // precede a real item inside any digit run
        const uint32_t d = rs_digit(key[r], shift, dmask);
        unsigned peers;
        uint32_t old;
        if constexpr (kOrMask) {
            // MATCH.ANY costs one step per DISTINCT value in the warp (ncu: the ADU pipe at 78 % on the passes over evenly
            // spread digits, which ran 1.7x longer than the pass over the clustered top digit).  The lanes OR their bit
            // into the digit's mask word instead: one shared-memory atomic whatever the digits are.
            atomicOr(&wm[d], 1u << lane);
            __syncwarp();
            peers = wm[d];
            old = wc[d];                                  // every peer reads mask and counter (broadcast) ...
            __syncwarp();
            if ((peers & lt) == 0u) {                     // ... then the lowest peer bumps the counter and clears the mask
                wc[d] = (uint16_t)(old + __popc(peers));
                wm[d] = 0u;
            }
            __syncwarp();
        } else {
            peers = __match_any_sync(kFull, d);
            old = wc[d];                                  // every peer reads the counter (broadcast) ...
            __syncwarp();
            if ((peers & lt) == 0u) wc[d] = (uint16_t)(old + __popc(peers));   // ... then the lowest peer bumps it
            __syncwarp();
        }
        const uint32_t rnk = old + __popc(peers & lt);
        if (r & 1) rk[r >> 1] |= rnk << 16; else rk[r >> 1] = rnk;
    }
    // values are only needed for the exchange below: load them now so the latency hides behind the scans
    uint32_t val[kRsItems];
    if (iota) {
#pragma unroll
        for (int r = 0; r < kRsItems; ++r) val[r] = beg + wbase + r * 32 + lane;
    } else {
        const uint32_t* vp = vin + wbase + lane;
        if (full) {
#pragma unroll
            for (int r = 0; r < kRsItems; ++r) val[r] = vp[r * 32];
        } else {
#pragma unroll
            for (int r = 0; r < kRsItems; ++r) val[r] = (wbase + r * 32 + lane < n) ? vp[r * 32] : 0u;
        }
    }
    __syncthreads();
    // per digit: exclusive prefix over warps, tile total
    uint32_t run[kRsBpt];
#pragma unroll
    for (int q = 0; q < kRsBpt; ++q) {
        uint32_t acc = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const uint32_t c = cnt[w * kRsBins + b0 + q];
            cnt[w * kRsBins + b0 + q] = (uint16_t)acc;
            acc += c;
        }
        run[q] = acc;
    }
    // publish, look back (padding only ever inflates the highest digit)
    uint32_t prefix[kRsBpt];
    {
        StT* st = status + ((size_t)s * tiles_ub + t) * kRsBins + b0;
#pragma unroll
        for (int q = 0; q < kRsBpt; ++q) {
            prefix[q] = 0;
            if ((uint32_t)(b0 + q) < nb) {
                uint32_t real = run[q];
                if ((uint32_t)(b0 + q) == nb - 1u) real -= (kRsTile - ntile);
                st_status(st + q, (t == 0 ? kGlobal : kLocal) | (StT)real);
            }
        }
        if (t > 0) {
#pragma unroll
            for (int q = 0; q < kRsBpt; ++q) {
                if ((uint32_t)(b0 + q) >= nb) continue;
                uint32_t real = run[q];
                if ((uint32_t)(b0 + q) == nb - 1u) real -= (kRsTile - ntile);
                // The tiles of a segment start together, so most predecessors are still LOCAL when a tile looks back and
                // the walk is long: kLb status words are loaded per step (independent loads, one L2 round trip).
                constexpr int kLb = 8;
                const StT* pst = st + q - kRsBins;
                StT pf = 0;
                bool done = false;
                for (uint32_t back = t; back > 0 && !done;) {
                    const uint32_t m = min(back, (uint32_t)kLb);
                    StT v[kLb];
#pragma unroll
                    for (int j = 0; j < kLb; ++j) v[j] = (uint32_t)j < m ? ld_status(pst - (size_t)j * kRsBins) : kGlobal;
#pragma unroll
                    for (int j = 0; j < kLb; ++j) {
                        if (done) continue;
                        while ((v[j] >> kFlagShift) == 0u) { __nanosleep(32); v[j] = ld_status(pst - (size_t)j * kRsBins); }
                        pf += v[j] & kCountMask;
                        if ((v[j] >> kFlagShift) == 2u) done = true;
                    }
                    back -= m;
                    pst -= (size_t)m * kRsBins;
                }
                prefix[q] = (uint32_t)pf;   // < 2^32: a segment holds fewer than 2^32 items
                st_status(st + q, kGlobal | (pf + real));
            }
        }
    }
    {
        uint32_t tot;
        uint32_t rsum = 0;
#pragma unroll
        for (int q = 0; q < kRsBpt; ++q) rsum += run[q];
        uint32_t ds = block_excl_scan(rsum, s_scan, tot);
#pragma unroll
        for (int q = 0; q < kRsBpt; ++q) {
            gbase[b0 + q] = dbase[q] + prefix[q] - ds;
            // fold the digit's tile-local start into every warp's prefix: one lookup per item in the exchange
#pragma unroll
            for (int w = 0; w < kWarps; ++w) cnt[w * kRsBins + b0 + q] += (uint16_t)ds;
            ds += run[q];
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kRsItems; ++r) {
        const uint32_t d = rs_digit(key[r], shift, dmask);
        const uint32_t pos = (uint32_t)wc[d] + ((rk[r >> 1] >> ((r & 1) * 16)) & 0xffffu);
        RsPair<KeyT> pr;
        pr.k = key[r]; pr.v = val[r];
        s_pairs[pos] = pr;
    }
    __syncthreads();
    if (full) {
#pragma unroll
        for (int r = 0; r < kRsItems; ++r) {
            const uint32_t i = r * kThreads + threadIdx.x;
            const RsPair<KeyT> pr = s_pairs[i];
            const uint32_t g = gbase[rs_digit(pr.k, shift, dmask)] + i;
            kout[g] = pr.k;
            vout[g] = pr.v;
        }
    } else {
        for (uint32_t i = threadIdx.x; i < ntile; i += kThreads) {
            const RsPair<KeyT> pr = s_pairs[i];
            const uint32_t g = gbase[rs_digit(pr.k, shift, dmask)] + i;
            kout[g] = pr.k;
            vout[g] = pr.v;
        }
    }
}

}  // namespace o3r
