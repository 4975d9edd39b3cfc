// host_bucket.cuh — host side of the fused bucket engine (bucket.cuh): per-frame bucket grids from a conservative bound of
// the frame's world bbox, buffer sizing, the launch sequence of one chunk of frames, the read-back and the verdict on it, and
// the steps both fused engines share (host_tile.cuh includes this file)
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "host_merge.cuh"

namespace {

// what a fused engine makes of its batch once the read-back has landed
enum class Verdict { ACCEPT, RERUN, NEXT_ENGINE };

// the batch's fills and sizing common to both fused engines (after the engine's own buffers are sized)
int fused_prepare(o3r_ctx* ctx, size_t cap_batch) {
    if (ctx->keep_frame_voxels) CU(ctx->vox.ensure(cap_batch * 16));
    FILL(ctx->counters.as<uint32_t>() + CNT_CELLBB, 24, FILL_CELLBB);
    ZERO(ctx->counters.as<uint32_t>() + CNT_PART, 8);
    ctx->tiled_now = false;
    return O3R_OK;
}

constexpr int kBkStrayCap = 8192;   // stray records per chunk (a couple per frame in practice)

inline long long floordiv_ll(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// Conservative world-space bounds of everything createSingleImgPtCloud can emit for this frame.  With the rectified-stereo Q
// (ctx->canon) a camera-frame point is ((q0 x + q3) s, (q5 y + q7) s, q11 s) with s = 1 / (q14 d + q15): for d in
// (min_disparity, d_max] the set is a frustum, i.e. inside the convex hull of its 8 corners, and a rigid transform keeps
// that.  Returns false when no bound exists (w changes sign over the disparity range) or the grid would be too large.
bool bk_frame_grid(const o3r_ctx* ctx, const float* T, int disp_type, bool label_mode, BkFrame& out, size_t& n_buckets) {
    const o3r_params& p = ctx->p;
    if (!ctx->canon) return false;
    const double* Q = p.Q;
    double dmax = INFINITY;
    if (!label_mode) {
        if (disp_type == O3R_DISP_U8) dmax = 255.0;
        else if (disp_type == O3R_DISP_U16) dmax = 65535.0 / p.disp_divisor;
    }
    const double wl = Q[14] * p.min_disparity + Q[15];
    double wh;
    if (std::isfinite(dmax)) wh = Q[14] * dmax + Q[15];
    else wh = Q[14] > 0 ? INFINITY : (Q[14] < 0 ? -INFINITY : wl);
    if (!(wl != 0.0) || !std::isfinite(wl) || (wl > 0) != (wh > 0) || wh == 0.0) return false;
    const double s_a = 1.0 / wl, s_b = std::isfinite(wh) ? 1.0 / wh : 0.0;
    const int xlo = p.cols_start_aft_cutout, xhi = p.cols - p.bounding_box - 1;
    const int ylo = p.bounding_box, yhi = p.rows - p.bounding_box - 1;
    if (xhi < xlo || yhi < ylo) return false;
    double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int c = 0; c < 8; ++c) {
        const double s = (c & 1) ? s_a : s_b;
        const double v0 = Q[0] * ((c & 2) ? xhi : xlo) + Q[3], v1 = Q[5] * ((c & 4) ? yhi : ylo) + Q[7];
        const double cam[3] = {v0 * s, v1 * s, Q[11] * s};
        for (int a = 0; a < 3; ++a) {
            const double w = (double)T[4 * a] * cam[0] + (double)T[4 * a + 1] * cam[1] + (double)T[4 * a + 2] * cam[2] + (double)T[4 * a + 3];
            if (!std::isfinite(w)) return false;
            mn[a] = std::min(mn[a], w); mx[a] = std::max(mx[a], w);
        }
    }
    long long lo[3], hi[3];
    for (int a = 0; a < 3; ++a) {
        const double pad = 1e-5 * std::max(std::fabs(mn[a]), std::fabs(mx[a])) + 1e-6;
        const double cl = std::floor((mn[a] - pad) * (double)ctx->inv_f) - 2, ch = std::floor((mx[a] + pad) * (double)ctx->inv_f) + 2;
        if (!(std::fabs(cl) < 8e6) || !(std::fabs(ch) < 8e6)) return false;   // float cell arithmetic stays exact below 2^23
        lo[a] = (long long)cl; hi[a] = (long long)ch;
    }
    const long long I0 = floordiv_ll(lo[0], kBkB), I1 = floordiv_ll(hi[0], kBkB);
    const long long J0 = floordiv_ll(lo[1], kBkB), J1 = floordiv_ll(hi[1], kBkB);
    const long long ni = I1 - I0 + 1, nj = J1 - J0 + 1;
    if (ni <= 0 || nj <= 0 || ni * nj > (1ll << 24)) return false;
    if (hi[2] - lo[2] >= (1ll << kBkKBits)) return false;
    out.i0c = (int)(I0 * kBkB); out.j0c = (int)(J0 * kBkB);
    out.ni = (int)ni; out.nj = (int)nj; out.k0 = (int)lo[2];
    out.base = 0; out.pad0 = out.pad1 = 0;
    n_buckets = (size_t)(ni * nj);
    return true;
}

struct BkPlan {
    std::vector<BkFrame> fr;          // per frame of the batch; base is relative to the frame's chunk
    std::vector<size_t> chunk_nb;     // buckets per chunk
    size_t max_chunk_nb = 0, total_nb = 0;
};

// bucket grids of all frames of the batch; false = the engine does not apply to this batch
bool bk_plan(const o3r_ctx* ctx, const o3r_frame* frames, int n, int chunk, int disp_type, bool label_mode, BkPlan& pl) {
    pl.fr.resize(n);
    pl.chunk_nb.clear();
    pl.max_chunk_nb = pl.total_nb = 0;
    for (int f0 = 0; f0 < n; f0 += chunk) {
        size_t at = 0;
        for (int i = f0; i < std::min(n, f0 + chunk); ++i) {
            size_t nb = 0;
            if (!bk_frame_grid(ctx, frames[i].T, disp_type, label_mode, pl.fr[i], nb)) return false;
            pl.fr[i].base = (uint32_t)at;
            at += nb;
            if (at >= (1ull << 28)) return false;
        }
        at = (at + 7) & ~(size_t)7;
        pl.chunk_nb.push_back(at);
        pl.max_chunk_nb = std::max(pl.max_chunk_nb, at);
        pl.total_nb += at;
    }
    return true;
}

// misc layout: [0..1] flags (upstream, reduce), [2..3] totals {points, non-empty buckets}, [4] scan ticket, [5] reduce ticket,
// [6] stray count, [7] debug voxel count (batch-wide), [64..64+n) per-frame voxel counts, then n bytes of per-frame pass-through flags
struct BkMisc {
    uint32_t *flags, *totals, *t_scan, *t_reduce, *dbg_cnt, *stray_cnt, *fvox;
    uint8_t* pass;
};
BkMisc bk_misc(o3r_ctx* ctx, int n) {
    uint32_t* m = ctx->bk_misc.as<uint32_t>();
    return BkMisc{m, m + 2, m + 4, m + 5, m + 7, m + 6, m + 64, reinterpret_cast<uint8_t*>(m + 64 + n)};
}

// sizes the engine's buffers for a batch and queues its fills
int bk_prepare(o3r_ctx* ctx, const BkPlan& pl, int n, size_t cap_batch, size_t cap_chunk) {
    CU(ctx->bk_frames.ensure((size_t)n * sizeof(BkFrame)));
    { int rcu = upload_small(ctx, ctx->bk_frames.p, pl.fr.data(), (size_t)n * sizeof(BkFrame)); if (rcu) return rcu; }
    CU(ctx->bk_counts.ensure(pl.max_chunk_nb * 4 + 64));
    const size_t nl_ub = std::min(pl.max_chunk_nb, cap_chunk);
    CU(ctx->bk_nl.ensure(nl_ub * 16 + 64));
    CU(ctx->bk_pts.ensure(cap_chunk * 16));
    CU(ctx->bk_pos.ensure(cap_chunk * 8));   // ordering keys (leaf key | scan position)
    CU(ctx->bk_status.ensure(((size_t)cdiv(pl.max_chunk_nb, kBkScanTile) + 1) * 8 + 64));
    CU(ctx->bk_stray.ensure((size_t)kBkStrayCap * sizeof(o3r_cell)));
    CU(ctx->bk_misc.ensure(256 + (size_t)n * 4 + (size_t)n));
    // every partial cell holds at least one point, and a bucket emits at most kBkMaxPart of them
    const size_t part_ub = std::min(cap_batch, pl.total_nb) + (size_t)kBkStrayCap * pl.chunk_nb.size();
    CU(ctx->partials.ensure(std::max<size_t>(part_ub, 1) * sizeof(o3r_cell)));
    CU(ctx->bbox.ensure((size_t)n * 6 * 4));
    const int rc = fused_prepare(ctx, cap_batch);
    if (rc) return rc;
    const BkMisc M = bk_misc(ctx, n);
    ZERO(M.flags, 8);
    ZERO(M.dbg_cnt, 4);
    return O3R_OK;
}

// one chunk of frames [f0, f0 + nc) through hist -> scan -> scatter -> reduce; partial cells are appended to ctx->partials at
// the device-side base cnt[CNT_PART] (advanced here)
template <int DT>
int bk_run_chunk(o3r_ctx* ctx, const AParams& P, const BkPlan& pl, int ci, int f0, int nc, int n, size_t cap_chunk) {
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const BkMisc M = bk_misc(ctx, n);
    const size_t nb = pl.chunk_nb[ci];
    const FrameDev* fr = ctx->d_frames.as<FrameDev>() + f0;
    const BkFrame* bk = ctx->bk_frames.as<BkFrame>() + f0;
    const uint32_t scan_tiles = cdiv(nb, kBkScanTile);
    const size_t nl_ub = std::min(nb, cap_chunk);
    unsigned long long* st_scan = ctx->bk_status.as<unsigned long long>();
    ZERO(ctx->bk_counts.p, nb * 4);
    ZERO(ctx->bk_status.p, ((size_t)scan_tiles + 1) * 8);
    ZERO(M.totals, 20);   // totals, both tickets, stray count
    ZERO(cnt + CNT_PARTCHUNK, 4);
    const dim3 grid(P.tiles_per_frame, nc);
    uint32_t* bbox = ctx->bbox.as<uint32_t>() + (size_t)f0 * 6;
    FILL(bbox, (size_t)(nc) * 24, FILL_BBOX);
    LAUNCH_N("k_bk_hist", (k_bk_hist<DT>), grid, kThreads, 0, P, fr, bk, ctx->inv_f, ctx->bk_counts.as<uint32_t>(), bbox, M.flags);
    LAUNCH(k_bk_frames, cdiv(nc, 64), 64, 0, nc, bbox, ctx->inv_f, M.pass + f0, M.fvox + f0);
    LAUNCH(k_bk_scan, scan_tiles, kThreads, 0, ctx->bk_counts.as<uint32_t>(), (uint32_t)nb, bk, M.pass + f0, nc,
           ctx->bk_nl.as<uint4>(), st_scan, M.t_scan, M.totals, M.flags);
    LAUNCH_N("k_bk_scatter", (k_bk_scatter<DT>), grid, kThreads, 0, P, fr, bk, M.pass + f0, ctx->inv_f,
             ctx->bk_counts.as<uint32_t>(), ctx->bk_pts.as<float4>(), ctx->bk_pos.as<unsigned long long>(), M.flags);
    const uint32_t rgrid = std::max(1u, std::min<uint32_t>(cdiv(nl_ub, kRdG), 148 * 4));
    float4* dbg = ctx->keep_frame_voxels ? ctx->vox.as<float4>() : nullptr;
    LAUNCH(k_bk_reduce, rgrid, kThreads, bk_reduce_smem(), ctx->bk_pts.as<float4>(), ctx->bk_pos.as<unsigned long long>(),
           ctx->bk_nl.as<uint4>(), M.totals, ctx->inv_c, ctx->inv_cz, ctx->partials.as<o3r_cell>(),
           cnt + CNT_PART, M.stray_cnt, (uint32_t)kBkStrayCap, M.t_reduce, M.fvox + f0, reinterpret_cast<int*>(cnt + CNT_CELLBB),
           M.flags, dbg, M.dbg_cnt);
    LAUNCH(k_bk_strays, 1, 1024, 0, ctx->partials.as<o3r_cell>(), cnt + CNT_PART, M.totals, M.stray_cnt, (uint32_t)kBkStrayCap,
           ctx->bk_stray.as<o3r_cell>(), cnt + CNT_PARTCHUNK, M.flags);
    LAUNCH(k_add_u32, 1, 32, 0, cnt + CNT_PART, cnt + CNT_PARTCHUNK);
    return O3R_OK;
}

// queues the copies of the per-frame voxel COUNTS (h_offs[1..n]) and the two overflow flag words (h_offs[n+1..n+2])
int bk_read_back(o3r_ctx* ctx, int n) {
    const BkMisc M = bk_misc(ctx, n);
    CU(cudaMemcpyAsync(ctx->h_offs + 1, M.fvox, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(ctx->h_offs + n + 1, M.flags, 8, cudaMemcpyDeviceToHost, ctx->st));
    return O3R_OK;
}

// on the landed read-back: a bucket too full / a point outside the grid bound sends this batch and the context's later ones
// to the sort engine
Verdict bk_verdict(o3r_ctx* ctx, int n) {
    const uint32_t* h = ctx->h_offs;
    if (!(h[n + 1] | h[n + 2])) return Verdict::ACCEPT;
    if (trace_on()) fprintf(stderr, "[o3r trace] bucket engine overflow flags %u %u: falling back to the sort engine\n", h[n + 1], h[n + 2]);
    ctx->bucket_off = true;
    return Verdict::NEXT_ENGINE;
}

}  // namespace
