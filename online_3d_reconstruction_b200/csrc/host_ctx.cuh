// host_ctx.cuh — the context (device buffers, streams, counters), the launch / error macros and the small helpers every host routine uses
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "blur.cuh"
#include "bucket.cuh"
#include "common.cuh"
#include "prepass.cuh"
#include "prereduce.cuh"
#include "sor.cuh"
#include "sort.cuh"
#include "stage_a.cuh"
#include "voxel.cuh"

using namespace o3r;

namespace {

std::string g_create_err;

inline double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
// O3R_TRACE set: host-side phase times go to stderr
inline bool trace_on() { static const bool on = getenv("O3R_TRACE") != nullptr; return on; }
struct Tr {
    bool on; double t; const char* where;
    explicit Tr(const char* w) : on(trace_on()), t(now_ms()), where(w) {}
    void mark(const char* what) { if (!on) return; const double n = now_ms(); fprintf(stderr, "[o3r trace] %s/%s %.3f ms\n", where, what, n - t); t = n; }
};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {   // (frees what this held: a record is reset by assigning a fresh one)
        if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
    cudaError_t ensure(size_t bytes, cudaStream_t st = nullptr, size_t preserve = 0) {
        if (bytes <= cap) return cudaSuccess;
        size_t want = std::max(bytes, cap + cap / 2);
        want = (want + 255) & ~(size_t)255;
        void* np = nullptr;
        cudaError_t e = cudaMalloc(&np, want);
        if (e != cudaSuccess) return e;
        if (p && preserve) {
            e = cudaMemcpyAsync(np, p, preserve, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { cudaFree(np); return e; }
        }
        if (p) cudaFree(p);
        p = np;
        cap = want;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// Small device fills (zeroed counters and tables, bbox / cell-range initial values) are not launched one by one: they queue up
// in the context and leave as ONE kernel in front of the next stream operation (every launch and CUDA / NCCL call of the
// library goes through LAUNCH / CU / NC, which flush the queue first), so stream order is what it would have been with
// separate kernels.  api() selects the context's device before anything is queued or flushed, and flushes what is left
// before the call returns: no fill outlives the call that queued it.
constexpr int kFillMax = 16;   // fills per flush: enough for every fill a fused cycle queues in front of its first kernel
struct FillList { uint32_t* p[kFillMax]; unsigned long long words[kFillMax]; int kind[kFillMax]; int n; };
enum { FILL_ZERO = 0, FILL_BBOX = 1, FILL_CELLBB = 2 };   // bbox: {~0, ~0, ~0, 0, 0, 0} per 6 words; cell range: {INT_MAX x3, INT_MIN x3}
struct FillQueue {
    FillList L{};
    size_t max_words = 0;
    void add(void* p, size_t bytes, int kind) {
        if (!bytes) return;
        L.p[L.n] = reinterpret_cast<uint32_t*>(p); L.words[L.n] = (bytes + 3) / 4; L.kind[L.n] = kind;
        max_words = std::max<size_t>(max_words, L.words[L.n]);
        ++L.n;
    }
    void clear() { L.n = 0; max_words = 0; }
};

enum { CNT_PTS = 0, CNT_VOX = 1, CNT_CYC = 2, CNT_NEW = 3, CNT_EMIT = 4, CNT_NEWSCAN = 5, CNT_BASE = 6, CNT_NRES = 7, CNT_ZERO = 8, CNT_PART = 9, CNT_PARTCHUNK = 10,
       CNT_XFLAG = 11, CNT_XRECV = 12, CNT_CHG0 = 13 /* and 14: the pending set's count, one per buffer */,
       CNT_CELLBB = 16, CNT_CHGOUT = 22, CNT_CHGERR = 23, CNT_N = 32 };

// engine of the merged path that served a batch; the values are what o3r_last_batch_engine returns
enum class Engine { SORT = 0, BUCKET = 1, TILE = 2 };

// ---- the context's records --------------------------------------------------------------------------------------------
// Between calls, only these records carry state; each frees what it holds.  Declared here (o3r_ctx holds them by value and
// every host_*.cuh needs it complete); each comment names the code that owns and writes the record.

// The last batch (host_frames.cuh): what the last o3r_frame_cloud / o3r_frames_cloud[_dev] call produced, read by
// o3r_last_batch_* and by a pending o3r_exchange_cycle.  No other call writes it or its payload buffers.
struct LastBatch {
    int n = 0;                        // frames
    size_t total = 0;                 // points (or per-frame voxels) of all frames, off[n]
    std::vector<uint32_t> off;        // per-frame offsets into pts / vox
    bool is_vox = false;              // the payload is per-frame voxels (vox), not points (pts)
    bool has_cellbb = false;          // cellbb = {imin, jmin, kmin, imax, jmax, kmax} of the payload's combined-grid cells
    int cellbb[6] = {0, 0, 0, 0, 0, 0};
    bool has_partials = false;        // TILED / FUSED: the batch also stands as n_part partial cells in `partials`
    size_t n_part = 0;
    Engine engine = Engine::SORT;     // not SORT: the batch materialised no per-frame clouds
    // payload; the sort engine also uses pts as its chunk scratch, the fused engines size partials / vox in their *_prepare
    DevBuf pts, vox, partials;
    uint32_t* h_offs = nullptr;       // pinned read-back of the offsets and the engines' flag words
    size_t h_offs_cap = 0;
    void clear() {
        n = 0; total = 0; off.clear(); is_vox = false; has_cellbb = false; has_partials = false; n_part = 0;
        engine = Engine::SORT;
    }
    ~LastBatch() { if (h_offs) cudaFreeHost(h_offs); }
};

// The resident map (host_merge.cuh): accumulators (ACCUMULATE) or points (RETAIN / dont_downsample).
struct Resident {
    DevBuf keys[2], acc[2], rgb[2];   // double-buffered: a merge writes the other set
    int cur = 0;
    // The exact cell count lives on the device (counters[CNT_NRES]); the host keeps an upper bound that is enough to size
    // buffers and launches, and tightens it from an asynchronous read-back of the previous merge.
    size_t n_ub = 0;
    bool n_exact = true;
    uint32_t* h_n = nullptr;          // pinned
    cudaEvent_t ev_n = nullptr;
    DevBuf cloud;                     // RETAIN / dont_downsample: the points
    size_t n_cloud = 0;
    ~Resident() { if (h_n) cudaFreeHost(h_n); if (ev_n) cudaEventDestroy(ev_n); }
};

// Change tracking of the resident map (host_changes.cuh); the context holds one exactly while tracking is on.  The pending
// set D (sorted unique absolute cell keys, double-buffered, count in counters[CNT_CHG0 + cur], host upper bound ub) or
// "everything" after an enable; the last emitted result (m records in out / okeys / ocnt), valid until the tracked state
// changes.
struct ChangeTracking {
    bool all = false, valid = false;
    int cur = 0;
    size_t ub = 0, m = 0;
    DevBuf keys[2], cnt, off, part, pos, out, okeys, ocnt;
};

// The accumulate exchange of a communicator (host_comm.cuh); o3r_comm_destroy replaces it with a fresh one.
struct Exchange {
    uint32_t slot_cap = 0;            // cells per (source, destination) slot
    DevBuf send, recv, list;
    bool pending_check = false;       // exchanges ran since the overflow flag was last reported
};

// The sharded RETAIN form of the exchange (host_retain.cuh): the points stay on the rank that made them; per appended frame
// its first point in the local cloud, its cycle and its global frame index (the order tag of cloud_big order); the last
// collective result.  o3r_comm_destroy replaces it with a fresh one; reset() forgets the cloud's history, not the buffers.
struct RetainShard {
    struct Frame { size_t first; uint32_t cycle, frame; };
    std::vector<Frame> frames;
    uint32_t cycles = 0;              // o3r_frames_cloud* calls since the communicator came (or the last clear)
    bool valid = false;               // out holds the result for the current local cloud
    size_t m = 0;
    size_t ftab_n = 0;                // frame records already in ftab
    DevBuf agree, ftab, tags, send, recv, pts, out;
    void reset() { frames.clear(); cycles = 0; valid = false; m = 0; ftab_n = 0; }
};

// The fused tile engine (host_tile.cuh): look-back words; flags / ticket / per-frame counts / pass-through guesses, and the
// engine policy the context's batches have taught it.
struct TileState {
    DevBuf tiles, misc, scratch;      // per-tile {count, scratch position, offset}; flags / counters; records in arrival order
    size_t scratch_cap = 0, part_cap = 0;   // records the scratch list / the batch's partial list hold (grown on overflow)
    bool off = false;                 // a batch exceeded the engine's limits: the bucket / sort engine serve this context from then on
    int R = -1;                       // window radius in use (-1: not chosen yet)
    int guess = -1;                   // PCL's overflow guard on the last frame seen (-1: none yet) = the guess for the next batch
    const uint8_t* guess_at = nullptr;   // where in `misc` the last uploaded per-frame guesses lie, and what they are
    std::vector<uint8_t> guess_dev;
    uint32_t attr = 0;                // k_tv instantiations whose shared-memory attribute is set
};

// The fused bucket engine (host_bucket.cuh): per-frame bucket grids, bucket counters / cursors, non-empty bucket list, binned
// points + scan positions, look-back words, flags / totals / tickets / per-frame counts, stray records.
struct BucketState {
    DevBuf frames, counts, nl, pts, pos, status, misc, stray;
    bool off = false;                 // a batch overflowed the engine's limits: the sort engine serves this context from then on
};

// The sort engine's tile pre-reduction in TILED mode (host_frames.cuh): skipped while it does not reduce (probed again every
// 16th batch); `now`: the running batch pre-reduces; status: its look-back words.
struct PreReduce { unsigned poor = 0, batches = 0; bool now = false; DevBuf status; };

// Input staging of the host-pointer frame path (host_frames.cuh), double-buffered: a prefetch of the next cycle's inputs
// fills one set while the kernels read the other.
struct InputStaging {
    struct Set { DevBuf disp, bgr, labels, coef, kp; } stg[2];
    struct Prefetch {                   // one record per staging set
        bool valid = false;
        int n = 0, disp_type = 0;
        uint64_t seq = 0;               // issue order (the older record is recycled when both are pending)
        std::vector<const void*> sig;   // host pointers of the prefetched frames
        cudaEvent_t ev = nullptr;
    } prefetch[2];
    uint64_t prefetch_seq = 0;
    // A prefetch request is only RECORDED by o3r_frames_prefetch; its ~2 memcpy calls per frame are issued by the next
    // frame-path call right after that call's kernels are queued (the GPU computes while the host issues copies)
    // instead of in front of them with the GPU idle.
    struct Deferred { bool pending = false; std::vector<o3r_frame> frames; int disp_type = 0; } deferred;
    // a staging set that holds no pending prefetch (inputs of finished calls are free: every frame-path call returns
    // only after its last input-reading kernel has completed)
    int busy_set = -1;   // staging set the queued kernels of the running frame-path call still read
    int free_stage_set() {
        if (busy_set >= 0) { prefetch[busy_set ^ 1].valid = false; return busy_set ^ 1; }
        if (!prefetch[0].valid) return 0;
        if (!prefetch[1].valid) return 1;
        const int s = prefetch[0].seq < prefetch[1].seq ? 0 : 1;
        prefetch[s].valid = false;
        return s;
    }
    int chunk_frames = 10, chunk_frames_dev = 1 << 30;   // frames per launch sequence (host / device inputs)
    std::vector<cudaEvent_t> chunk_ev;
    cudaEvent_t chunk_event(size_t i) {
        while (chunk_ev.size() <= i) {
            cudaEvent_t e;
            cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
            chunk_ev.push_back(e);
        }
        return chunk_ev[i];
    }
    DevBuf frames;                      // the batch's FrameDev descriptors
    ~InputStaging() {
        for (auto& pf : prefetch) if (pf.ev) cudaEventDestroy(pf.ev);
        for (auto e : chunk_ev) cudaEventDestroy(e);
    }
};

// StatisticalOutlierRemoval (host_sor.cuh): the kept points and their offsets (pts / off), the distances and thresholds, and
// the grid / sort scratch of sor_filter
struct SorScratch { DevBuf hard, pts, off, dist, grids, pgrids, rows, thr, skeys, svals, cnt, cntoff, spts; };

// Blurs (o3r_blur_u8 and the frame path's blur_kernel): o3r_blur_u8's source plane, the blurred planes and jobs, and the
// bilateral LUTs (colour weights, space weights, per-row tap extents) of `kernel`, cached by bilateral_lut
struct Blur { DevBuf disp, out, jobs, lut; int kernel = -1, radius = 0, maxk = 0; };

// Registration against the resident map (host_register.cuh): the staged host points, the CTA partial sums, the iteration
// state on the device and its pinned read-back
struct Registration {
    DevBuf pts, part, state;
    void* h_state = nullptr;
    ~Registration() { if (h_state) cudaFreeHost(h_state); }
};

// Meshing of the resident map (host_mesh.cuh): per-tile vertex / triangle counts and offsets, the two totals and their pinned
// read-back, the resident position -> vertex map, and the result (vertices, normals, triangles) o3r_cloud_mesh_dev points at
struct Meshing {
    DevBuf vcnt, voff, tcnt, toff, tot, vmap, verts, normals, tris;
    uint32_t* h_tot = nullptr;
    ~Meshing() { if (h_tot) cudaFreeHost(h_tot); }
};

// The pre-pass (o3r_disp_variance / o3r_plane_fit in o3r_api.cu): plane fit / variance gate scratch
struct PrePass { DevBuf labels, disp, sums, rows, coef; };

// Optional per-kernel event timing (o3r_profile; bench.py's roofline leg)
struct Profiling {
    struct Rec { const char* name; cudaEvent_t a, b; };
    bool on = false;
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t get() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    ~Profiling() {
        for (auto& r : recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        for (auto e : pool) cudaEventDestroy(e);
    }
};

}  // namespace

struct o3r_ctx {
    o3r_params p;
    std::mutex mu;
    std::string err;
    uint64_t launches = 0;
    bool pdl_off = false;   // the next launch waits for the stream in full (set after NCCL calls, see LAUNCH_N)
    FillQueue fq;   // pending device fills (see FillList)
    cudaStream_t st = nullptr, st_copy = nullptr, st_copy2 = nullptr;   // two copy streams: the per-copy set-up gaps of one hide behind the other
    cudaEvent_t ev_copy2 = nullptr;
    DevBuf counters;
    uint32_t* h_counters = nullptr;   // pinned
    // set by o3r_create / o3r_set_keep_frame_voxels / o3r_comm_*
    int nx = 0, ny = 0;
    uint32_t npix = 0;
    int canon = 0;
    float leaf_f = 0, inv_f = 0, leaf_c = 0, inv_c = 0, inv_cz = 0;
    DevBuf lut_r, lut_z;
    bool keep_frame_voxels = false;   // parity probe: the fused engines also write every per-frame voxel centroid (any order)
    void* comm = nullptr;             // ncclComm_t (host_comm.cuh)
    bool comm_owned = false;
    int world = 1, rank = 0;

    LastBatch last;
    Resident res;
    std::unique_ptr<ChangeTracking> chg;
    Exchange x;
    RetainShard rt;
    TileState tv;
    BucketState bk;
    PreReduce pre;
    InputStaging in;
    SorScratch sor;
    Blur blur;
    PrePass pp;
    Registration reg;
    Meshing mesh;
    Profiling prof;

    // Shared per-call scratch: sized on demand and used by several paths within one call.  It holds nothing a later call
    // reads; the one exception is the result o3r_cloud_downsample_dev points at (in ckey or cacc), valid until the next call.
    DevBuf tile_cnt, tile_off, bbox, frame_off, grids, sortbuf, hist, plan_all, plan_v2, ghist;
    DevBuf head_cnt, head_off, vox_off, seg2, tmat, mask, runwork;
    DevBuf ckey, cacc, crgb, new_cnt, new_off, new_keys, okeys;   // a cycle's cell list and the merge's work buffers
    size_t n_cyc_ub = 0;              // cells of the cycle list built by the running call
    DevBuf in_pts, out_pts;           // caller points staged by o3r_voxel_grid / o3r_sor / o3r_cloud_append; o3r_voxel_grid's result
    DevBuf ck_cells, ck_res;          // checkpoints (host_checkpoint.cuh): packed / staged o3r_cell records, the import check's result

    bool retain() const { return p.dont_downsample || p.merge_mode == O3R_MERGE_RETAIN; }
    bool tiled() const { return !p.dont_downsample && (p.merge_mode == O3R_MERGE_ACCUMULATE_TILED || p.merge_mode == O3R_MERGE_ACCUMULATE_FUSED); }
    bool fused() const { return !p.dont_downsample && p.merge_mode == O3R_MERGE_ACCUMULATE_FUSED; }
    int fail(int code, const std::string& m) { err = m; return code; }
    int fail_cuda(cudaError_t e, const char* what, const char* file, int line) {
        const char* base = strrchr(file, '/');
        char buf[512];
        snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s [%s:%d]", (int)e, cudaGetErrorString(e), what, base ? base + 1 : file, line);
        err = buf;
        return O3R_ERR_CUDA;
    }
    // (o3r_destroy makes the device current and drains the streams first; the records and buffers free themselves after this)
    ~o3r_ctx() {
        if (h_counters) cudaFreeHost(h_counters);
        if (ev_copy2) cudaEventDestroy(ev_copy2);
        if (st_copy2) cudaStreamDestroy(st_copy2);
        if (st_copy) cudaStreamDestroy(st_copy);
        if (st) cudaStreamDestroy(st);
    }
};

int fill_flush(o3r_ctx* ctx);

#define CU(call)                                                              \
    do {                                                                      \
        if (ctx->fq.L.n) { int rcf_ = fill_flush(ctx); if (rcf_) return rcf_; } \
        cudaError_t e_ = (call);                                              \
        if (e_ != cudaSuccess) return ctx->fail_cuda(e_, #call, __FILE__, __LINE__);    \
    } while (0)

// Kernels go out with programmatic stream serialisation: the next kernel's launch overlaps the tail of the previous one,
// and its wait_prior() (common.cuh) restores the full dependency before it touches memory.  Copies and event records keep
// plain stream order.  The first launch of an API call and the first after an NCCL call go without it (ctx->pdl_off):
// kernels the library does not own (the caller's, NCCL's) do not promise to leave their trigger to their completion.
#define LAUNCH_N(name, kernel, grid, block, smem, ...)                        \
    do {                                                                      \
        if (ctx->fq.L.n) { int rcf_ = fill_flush(ctx); if (rcf_) return rcf_; } \
        cudaEvent_t pa_ = nullptr, pb_ = nullptr;                             \
        if (ctx->prof.on) {                                                   \
            pa_ = ctx->prof.get(); pb_ = ctx->prof.get();                     \
            cudaEventRecord(pa_, ctx->st);                                    \
        }                                                                     \
        cudaLaunchAttribute at_[1];                                           \
        at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;       \
        at_[0].val.programmaticStreamSerializationAllowed = ctx->pdl_off ? 0 : 1; \
        ctx->pdl_off = false;                                                 \
        cudaLaunchConfig_t cfg_ = {};                                         \
        cfg_.gridDim = dim3(grid); cfg_.blockDim = dim3(block);               \
        cfg_.dynamicSmemBytes = (smem); cfg_.stream = ctx->st;                \
        cfg_.attrs = at_; cfg_.numAttrs = 1;                                  \
        cudaError_t e_ = cudaLaunchKernelEx(&cfg_, kernel, __VA_ARGS__);      \
        ++ctx->launches;                                                      \
        if (e_ == cudaSuccess) e_ = cudaGetLastError();                       \
        if (e_ != cudaSuccess) return ctx->fail_cuda(e_, #kernel, __FILE__, __LINE__);  \
        if (pa_) {                                                            \
            cudaEventRecord(pb_, ctx->st);                                    \
            ctx->prof.recs.push_back({name, pa_, pb_});                       \
        }                                                                     \
    } while (0)
#define LAUNCH(kernel, grid, block, smem, ...) LAUNCH_N(#kernel, kernel, grid, block, smem, __VA_ARGS__)

namespace {

inline uint32_t cdiv(size_t a, size_t b) { return (uint32_t)((a + b - 1) / b); }

// Small host->device payloads (frame descriptors, segment bounds, plans) travel as KERNEL PARAMETERS, not through the
// copy engine: a pageable cudaMemcpyAsync on the compute stream would queue behind a 184 MB input prefetch that
// occupies the H2D engine, and the whole cycle would wait for it.
struct SmallBlob { uint32_t w[960]; };   // 3840 bytes (kernel parameters are limited to 4 KB)
__global__ void k_put_blob(uint32_t* __restrict__ dst, SmallBlob b, int n_words) {
    wait_prior();
    for (int i = threadIdx.x; i < n_words; i += blockDim.x) dst[i] = b.w[i];
}
int upload_small(o3r_ctx* ctx, void* dst, const void* src, size_t bytes) {
    const size_t cap = sizeof(SmallBlob);
    for (size_t at = 0; at < bytes; at += cap) {
        const size_t nb = std::min(cap, bytes - at);
        SmallBlob b;
        memcpy(b.w, (const char*)src + at, nb);
        if (nb % 4) memset((char*)b.w + nb, 0, 4 - nb % 4);
        LAUNCH(k_put_blob, 1, 256, 0, reinterpret_cast<uint32_t*>((char*)dst + at), b, (int)((nb + 3) / 4));
    }
    return O3R_OK;
}
// Fills run as kernels on the compute stream for the same reason: cudaMemsetAsync may be served by a copy engine and then
// queues behind an input prefetch.  `bytes` and `dst` are multiples of 4 (all callers fill u32 tables).
__global__ void __launch_bounds__(kThreads) k_fill_list(FillList L) {
    wait_prior();
    for (int r = 0; r < L.n; ++r) {
        uint32_t* dst = L.p[r];
        const size_t n_words = L.words[r], stride = (size_t)gridDim.x * kThreads;
        const size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x;
        if (L.kind[r] == FILL_ZERO) {
            const size_t n4 = ((uintptr_t)dst % 16 == 0) ? n_words / 4 : 0;
            uint4* d4 = reinterpret_cast<uint4*>(dst);
            for (size_t j = i; j < n4; j += stride) d4[j] = make_uint4(0u, 0u, 0u, 0u);
            for (size_t j = n4 * 4 + i; j < n_words; j += stride) dst[j] = 0u;
        } else if (L.kind[r] == FILL_BBOX) {
            for (size_t j = i; j < n_words; j += stride) dst[j] = (j % 6 < 3) ? 0xffffffffu : 0u;
        } else {
            for (size_t j = i; j < n_words; j += stride) dst[j] = (j % 6 < 3) ? 0x7fffffffu : 0x80000000u;
        }
    }
}
}  // namespace
int fill_flush(o3r_ctx* ctx) {
    if (!ctx->fq.L.n) return O3R_OK;
    const FillList L = ctx->fq.L;
    const uint32_t g = (uint32_t)std::min<size_t>((ctx->fq.max_words / 4 + kThreads - 1) / kThreads + 1, 148 * 8);
    ctx->fq.clear();   // (before the launch macro: it flushes a non-empty queue)
    LAUNCH_N("k_fill", k_fill_list, g, kThreads, 0, L);
    return O3R_OK;
}

// Every C-ABI entry point that takes a context runs its body through api(): under the context's lock, with the context's
// device current (a raw call: CU would flush queued fills first, while another device may still be current), and with
// whatever fills the body left queued flushed before it returns.  A failed body's code and message are what the call
// returns, whatever the flush does.
template <typename F>
int api(o3r_ctx* ctx, F&& body) {
    if (!ctx) return O3R_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    const cudaError_t e = cudaSetDevice(ctx->p.device);
    if (e != cudaSuccess) return ctx->fail_cuda(e, "cudaSetDevice(ctx->p.device)", __FILE__, __LINE__);
    ctx->pdl_off = true;   // the caller may have queued its own kernels on the stream since the last call (see LAUNCH_N)
    const int rc = body();
    if (!rc) return fill_flush(ctx);
    if (ctx->fq.L.n) { const std::string err = ctx->err; fill_flush(ctx); ctx->err = err; }
    return rc;
}

namespace {
int fill_queue(o3r_ctx* ctx, void* dst, size_t bytes, int kind) {
    if (bytes == 0) return O3R_OK;
    if (ctx->fq.L.n == kFillMax) { int rc = fill_flush(ctx); if (rc) return rc; }
    ctx->fq.add(dst, bytes, kind);
    return O3R_OK;
}
#define ZERO(ptr, bytes) do { int rcz_ = fill_queue(ctx, (ptr), (bytes), FILL_ZERO); if (rcz_) return rcz_; } while (0)
#define FILL(ptr, bytes, kind) do { int rcz_ = fill_queue(ctx, (ptr), (bytes), (kind)); if (rcz_) return rcz_; } while (0)
inline size_t disp_elem(int t) { return t == O3R_DISP_U8 ? 1 : t == O3R_DISP_U16 ? 2 : t == O3R_DISP_F32 ? 4 : 8; }
// calls f(std::integral_constant<int, DT>) for the runtime disparity type: the one place it becomes a template argument
template <typename F>
int with_disp_type(int disp_type, F&& f) {
    switch (disp_type) {
        case O3R_DISP_U8: return f(std::integral_constant<int, O3R_DISP_U8>());
        case O3R_DISP_U16: return f(std::integral_constant<int, O3R_DISP_U16>());
        case O3R_DISP_F32: return f(std::integral_constant<int, O3R_DISP_F32>());
        default: return f(std::integral_constant<int, O3R_DISP_F64>());
    }
}

int read_counters(o3r_ctx* ctx) {
    CU(cudaMemcpyAsync(ctx->h_counters, ctx->counters.p, CNT_N * 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    return O3R_OK;
}

// LUTs of cv::bilateralFilter(src, dst, d = k, sigmaColor = 2k, sigmaSpace = k/2) (pose_functions.cpp:1044), computed on the
// host with std::exp exactly as OpenCV 3.1 bilateralFilter_8u (and the oracle) do, cached per kernel size.
int bilateral_lut(o3r_ctx* ctx, int k, BilateralLut* out) {
    Blur& B = ctx->blur;
    if (B.kernel != k) {
        double sigma_color = (double)(k * 2), sigma_space = (double)(k / 2);
        if (sigma_color <= 0) sigma_color = 1;
        if (sigma_space <= 0) sigma_space = 1;
        const double gc = -0.5 / (sigma_color * sigma_color), gs = -0.5 / (sigma_space * sigma_space);
        const int radius = std::max(k <= 0 ? (int)std::lrint(sigma_space * 1.5) : k / 2, 1);
        std::vector<float> buf(256);
        for (int i = 0; i < 256; ++i) buf[i] = (float)std::exp(i * i * gc);
        std::vector<int> jm(2 * radius + 1, -1);
        for (int i = -radius; i <= radius; ++i)
            for (int j = -radius; j <= radius; ++j) {
                const double r = std::sqrt((double)i * i + (double)j * j);
                if (r > radius) continue;
                buf.push_back((float)std::exp(r * r * gs));
                jm[i + radius] = std::max(jm[i + radius], j);   // the mask is symmetric in j
            }
        const int maxk = (int)buf.size() - 256;
        const size_t bytes = buf.size() * 4 + jm.size() * 4;
        std::vector<unsigned char> blob(bytes);
        memcpy(blob.data(), buf.data(), buf.size() * 4);
        memcpy(blob.data() + buf.size() * 4, jm.data(), jm.size() * 4);
        CU(B.lut.ensure(bytes));
        { int rcu = upload_small(ctx, B.lut.p, blob.data(), bytes); if (rcu) return rcu; }
        B.kernel = k; B.radius = radius; B.maxk = maxk;
        CU(cudaFuncSetAttribute(k_bilateral, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bilateral_smem(radius, maxk)));
    }
    out->color_w = B.lut.as<float>();
    out->space_w = out->color_w + 256;
    out->jmax = reinterpret_cast<const int*>(out->space_w + B.maxk);
    out->radius = B.radius; out->maxk = B.maxk;
    return O3R_OK;
}

}  // namespace
