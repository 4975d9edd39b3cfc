// host_tile.cuh — host side of the fused tile engine (tile.cuh): the window bound, the pass-through guess, buffer sizing,
// the launch sequence of one chunk of frames, the read-back and the verdict on it (reruns, engine policy)
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "host_bucket.cuh"
#include "tile.cuh"

namespace {

// a batch's plan: the tiling and the window bound, and the pass-through guesses and window radius of the current attempt
struct TvPlan {
    int ntx = 0, nty = 0;
    size_t tiles_per_frame = 0;
    double L = 0;                    // pixels per unit of |q14 d + q15| that two points of one leaf can lie apart (tile.cuh, header)
    bool guess_pass = false;         // the guard's verdict on a nominal frame (first batch of a context)
    std::vector<uint8_t> guess;      // per frame: PCL's overflow guard as the tile kernel will assume it
    int R = 0;                       // 0: every frame is guessed to pass through (no window)
    double wlim(int R) const { return (double)(R + 1) / L; }
};

// inverse of the 3x3 part of a row-major 3x4 float matrix, in double; false when it is (numerically) singular
inline bool tv_inv3(const float* T, double inv[9]) {
    const double a = T[0], b = T[1], c = T[2], d = T[4], e = T[5], f = T[6], g = T[8], h = T[9], i = T[10];
    const double A = e * i - f * h, B = -(d * i - f * g), C = d * h - e * g;
    const double det = a * A + b * B + c * C;
    const double scale = std::fabs(a) + std::fabs(b) + std::fabs(c) + std::fabs(d) + std::fabs(e) + std::fabs(f) + std::fabs(g) +
                         std::fabs(h) + std::fabs(i);
    if (!std::isfinite(det) || !(std::fabs(det) > 1e-9 * scale * scale * scale)) return false;
    const double r = 1.0 / det;
    inv[0] = A * r; inv[1] = -(b * i - c * h) * r; inv[2] = (b * f - c * e) * r;
    inv[3] = B * r; inv[4] = (a * i - c * g) * r;  inv[5] = -(a * f - c * d) * r;
    inv[6] = C * r; inv[7] = -(a * h - b * g) * r; inv[8] = (a * e - b * d) * r;
    return true;
}

// Geometry of the tiling and of the window bound (tile.cuh, header).  false = the engine does not apply.
bool tv_plan(const o3r_ctx* ctx, const AParams& P, const o3r_frame* frames, int n, TvPlan& pl) {
    const o3r_params& p = ctx->p;
    if (!ctx->canon || !P.vec || P.kp_tiles != 0 || P.J != 1 || P.nx <= 0 || P.ny <= 0) return false;
    const double* Q = p.Q;
    if (Q[0] == 0.0 || Q[5] == 0.0 || Q[11] == 0.0) return false;
    pl.ntx = (P.nx + kTvW - 1) / kTvW;
    pl.nty = (P.ny + kTvH - 1) / kTvH;
    pl.tiles_per_frame = (size_t)pl.ntx * pl.nty;
    const int xlo = P.x0, xhi = P.x0 + P.nx - 1, ylo = P.bb, yhi = P.bb + P.ny - 1;
    const double tx = std::max(std::fabs(Q[0] * xlo + Q[3]), std::fabs(Q[0] * xhi + Q[3])) / std::fabs(Q[11]);
    const double ty = std::max(std::fabs(Q[5] * ylo + Q[7]), std::fabs(Q[5] * yhi + Q[7])) / std::fabs(Q[11]);
    // nominal depth range: disparities in (min_disparity, 2 min_disparity]
    const double w_a = Q[14] * p.min_disparity + Q[15], w_b = Q[14] * 2.0 * p.min_disparity + Q[15];
    if (!(w_a != 0.0) || !std::isfinite(w_a) || !std::isfinite(w_b) || (w_a > 0) != (w_b > 0)) return false;
    const double s_a = 1.0 / w_a, s_b = 1.0 / w_b;
    const double range = std::fabs(Q[11] * s_a) * std::sqrt(1.0 + tx * tx + ty * ty);
    double tmax = 0;
    for (int i = 0; i < n; ++i)
        for (int a = 0; a < 3; ++a) tmax = std::max(tmax, (double)std::fabs(frames[i].T[4 * a + 3]));
    if (!std::isfinite(tmax) || !std::isfinite(range)) return false;
    // Two points of one leaf differ by less than the leaf edge on every WORLD axis (plus the float rounding of the transformed
    // coordinates and of the cell function: a few ulps of the largest coordinate).  Back in the camera frame, dC = M^-1 dP:
    // |dX| <= edge * sum_a |M^-1[0][a]| and so on, and |x1 - x2| <= (|dX| + |t2| |dZ|) |w1| / |q0| (header of tile.cuh).
    const double edge = (double)ctx->leaf_f * 1.001 + 16.0 * FLT_EPSILON * (tmax + range);
    pl.L = 0;
    for (int i = 0; i < n; ++i) {
        double inv[9];
        if (!tv_inv3(frames[i].T, inv)) return false;
        const double sx = std::fabs(inv[0]) + std::fabs(inv[1]) + std::fabs(inv[2]);
        const double sy = std::fabs(inv[3]) + std::fabs(inv[4]) + std::fabs(inv[5]);
        const double sz = std::fabs(inv[6]) + std::fabs(inv[7]) + std::fabs(inv[8]);
        pl.L = std::max(pl.L, std::max((sx + tx * sz) / std::fabs(Q[0]), (sy + ty * sz) / std::fabs(Q[5])) * edge);
    }
    if (!std::isfinite(pl.L) || !(pl.L > 0)) return false;
    // the guard on a nominal frame: extents of the frustum slab, rotated by the first frame's matrix
    double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    const float* T = frames[0].T;
    for (int c = 0; c < 8; ++c) {
        const double s = (c & 1) ? s_a : s_b;
        const double cam[3] = {(Q[0] * ((c & 2) ? xhi : xlo) + Q[3]) * s, (Q[5] * ((c & 4) ? yhi : ylo) + Q[7]) * s, Q[11] * s};
        for (int a = 0; a < 3; ++a) {
            const double w = (double)T[4 * a] * cam[0] + (double)T[4 * a + 1] * cam[1] + (double)T[4 * a + 2] * cam[2];
            mn[a] = std::min(mn[a], w); mx[a] = std::max(mx[a], w);
        }
    }
    double cells = 1;
    for (int a = 0; a < 3; ++a) cells *= std::floor((mx[a] - mn[a]) * (double)ctx->inv_f) + 1.0;
    pl.guess_pass = cells > 2147483647.0;
    return true;
}

// false = the engine does not serve this batch; otherwise the first guesses and (once per context) the window radius
bool tv_begin(o3r_ctx* ctx, const AParams& P, const o3r_frame* frames, int n, TvPlan& pl) {
    if (ctx->tv.off || !tv_plan(ctx, P, frames, n, pl)) return false;
    pl.guess.assign(n, (uint8_t)(ctx->tv.guess >= 0 ? ctx->tv.guess : (pl.guess_pass ? 1 : 0)));
    if (ctx->tv.R < 0) {   // smallest window that covers the nominal depth range (disparities up to 2 min_disparity)
        const double w_need = std::fabs(ctx->p.Q[14] * 2.0 * ctx->p.min_disparity + ctx->p.Q[15]);
        ctx->tv.R = kTvMaxR;
        for (int r = 1; r <= kTvMaxR; ++r)
            if (pl.wlim(r) >= w_need) { ctx->tv.R = r; break; }
    }
    return true;
}

// misc layout (u32 words): [0] flags, [1] ticket, [2] debug voxel count, [3] scratch cursor, [4] largest cursor of the batch,
// [16 .. 16 + n) per-frame voxel counts, then n bytes of guessed and n bytes of actual pass-through flags
struct TvMisc {
    uint32_t *flags, *ticket, *dbg_cnt, *cursor, *max_cursor, *fvox;
    uint8_t *guess, *actual;
};
TvMisc tv_misc(o3r_ctx* ctx, int n) {
    uint32_t* m = ctx->tv.misc.as<uint32_t>();
    uint8_t* b = reinterpret_cast<uint8_t*>(m + 16 + n);
    return TvMisc{m, m + 1, m + 2, m + 3, m + 4, m + 16, b, b + n};
}

// The record lists are sized from what the previous batches needed (the device reports overflow, the host grows and reruns):
// a tile can emit up to kTvItems records, a typical one a few dozen.
int tv_prepare(o3r_ctx* ctx, TvPlan& pl, int n, int chunk, size_t cap_batch) {
    pl.R = std::all_of(pl.guess.begin(), pl.guess.end(), [](uint8_t g) { return g != 0; }) ? 0 : ctx->tv.R;
    const size_t tiles_chunk = pl.tiles_per_frame * (size_t)chunk, tiles_batch = pl.tiles_per_frame * (size_t)n;
    CU(ctx->tv.tiles.ensure(3 * (tiles_chunk + 4) * 4));
    CU(ctx->tv.misc.ensure((16 + (size_t)n) * 4 + 2 * (size_t)n + 16));
    CU(ctx->bbox.ensure((size_t)n * 6 * 4));
    const size_t hard_chunk = std::min(tiles_chunk * (size_t)kTvItems, pl.tiles_per_frame ? cap_batch / n * chunk : 0);
    const size_t hard_batch = std::min(tiles_batch * (size_t)kTvItems, cap_batch);
    ctx->tv.scratch_cap = std::min(std::max(ctx->tv.scratch_cap, tiles_chunk * 256), std::max<size_t>(hard_chunk, 1));
    ctx->tv.part_cap = std::min(std::max(ctx->tv.part_cap, tiles_batch * 256), std::max<size_t>(hard_batch, 1));
    if (ctx->tv.scratch_cap >= (1ull << 32) || ctx->tv.part_cap >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "batch too large for the tile engine");
    CU(ctx->tv.scratch.ensure(ctx->tv.scratch_cap * sizeof(o3r_cell)));
    CU(ctx->last.partials.ensure(ctx->tv.part_cap * sizeof(o3r_cell)));
    const TvMisc M = tv_misc(ctx, n);
    ZERO(M.flags, (16 + (size_t)n) * 4);   // (the guess bytes follow these words: the fill leaves them alone)
    if (ctx->tv.guess_at != M.guess || ctx->tv.guess_dev != pl.guess) {   // steady state: the device holds these guesses already
        const int rc = upload_small(ctx, M.guess, pl.guess.data(), (size_t)n);
        if (rc) return rc;
        ctx->tv.guess_at = M.guess;
        ctx->tv.guess_dev = pl.guess;
    }
    return fused_prepare(ctx, cap_batch);
}

template <int DT, int R>
int tv_launch(o3r_ctx* ctx, const AParams& P, const TvArgs& A, uint32_t n_tiles) {
    const uint32_t bit = 1u << (DT * (kTvMaxR + 1) + R);
    if (!(ctx->tv.attr & bit)) {   // (the attribute is per function and device)
        CU(cudaFuncSetAttribute(k_tv<DT, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tv_smem<R>()));
        cudaFuncSetAttribute(k_tv<DT, R>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        ctx->tv.attr |= bit;
    }
    LAUNCH_N("k_tv", (k_tv<DT, R>), n_tiles, kTvThreads, tv_smem<R>(), P, A);
    return O3R_OK;
}

// one chunk of frames [f0, f0 + nc): the fused kernel + the guard check; partial cells are appended to ctx->last.partials at the
// device-side base cnt[CNT_PART] (advanced here)
template <int DT>
int tv_run_chunk(o3r_ctx* ctx, const AParams& P, const TvPlan& pl, int f0, int nc, int n) {
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const TvMisc M = tv_misc(ctx, n);
    const uint32_t n_tiles = (uint32_t)(pl.tiles_per_frame * (size_t)nc);
    uint32_t* tile_cnt = ctx->tv.tiles.as<uint32_t>();
    uint32_t* tile_at = tile_cnt + (pl.tiles_per_frame * (size_t)nc + 4);
    uint32_t* tile_off = tile_at + (pl.tiles_per_frame * (size_t)nc + 4);
    ZERO(M.ticket, 4);
    ZERO(M.cursor, 4);
    ZERO(cnt + CNT_PARTCHUNK, 4);
    uint32_t* bbox = ctx->bbox.as<uint32_t>() + (size_t)f0 * 6;
    FILL(bbox, (size_t)(nc) * 24, FILL_BBOX);
    TvArgs A;
    A.frames = ctx->in.frames.as<FrameDev>() + f0;
    A.frame_pass = M.guess + f0;
    A.ntx = pl.ntx; A.nty = pl.nty; A.n_frames = nc;
    A.inv_f = ctx->inv_f; A.icx = ctx->inv_c; A.icz = ctx->inv_cz;
    A.wlim = pl.R > 0 ? pl.wlim(pl.R) : INFINITY;
    {   // the kernel's LUT path flags d > dlim_i: every live u8 disparity (thr_i, dlim_i] must keep |q14 d + q15| below the
        // bound.  Scan up from the first live one and stop at the first that breaks it: when |w| is not monotone over the live
        // range (q15 of the opposite sign to q14), disparities past that point are flagged even where |w| drops back below.
        int dl = std::max(P.thr_i, -1);
        for (int d = dl + 1; d < 256 && std::fabs(ctx->p.Q[14] * d + ctx->p.Q[15]) < A.wlim; ++d) dl = d;
        A.dlim_i = dl;
    }
    A.scratch = ctx->tv.scratch.as<o3r_cell>();
    A.scratch_cap = (uint32_t)ctx->tv.scratch_cap;
    A.cursor = M.cursor;
    A.tile_cnt = tile_cnt;
    A.tile_at = tile_at;
    A.ticket = M.ticket;
    A.frame_vox = M.fvox + f0;
    A.bbox = bbox;
    A.cellbb = reinterpret_cast<int*>(cnt + CNT_CELLBB);
    A.flags = M.flags;
    A.dbg_vox = ctx->keep_frame_voxels ? ctx->last.vox.as<float4>() : nullptr;
    A.dbg_cnt = M.dbg_cnt;
    int rc;
    switch (pl.R) {
        case 0: rc = tv_launch<DT, 0>(ctx, P, A, n_tiles); break;
        case 1: rc = tv_launch<DT, 1>(ctx, P, A, n_tiles); break;
        case 2: rc = tv_launch<DT, 2>(ctx, P, A, n_tiles); break;
        case 3: rc = tv_launch<DT, 3>(ctx, P, A, n_tiles); break;
        default: rc = tv_launch<DT, 4>(ctx, P, A, n_tiles); break;
    }
    if (rc) return rc;
    // tile order: offsets = scan of the per-tile counts, then one warp per tile copies its records behind the batch's list
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, tile_cnt, tile_off, n_tiles, cnt + CNT_PARTCHUNK);
    LAUNCH(k_tv_compact, cdiv(n_tiles, kWarps), kThreads, 0, ctx->tv.scratch.as<o3r_cell>(), tile_cnt, tile_at, tile_off, n_tiles,
           ctx->last.partials.as<o3r_cell>(), cnt + CNT_PART, cnt + CNT_PARTCHUNK, (uint32_t)ctx->tv.part_cap, M.cursor, M.max_cursor,
           M.flags, nc, bbox, ctx->inv_f, M.guess + f0, M.actual + f0);
    LAUNCH(k_add_u32, 1, 32, 0, cnt + CNT_PART, cnt + CNT_PARTCHUNK);
    return O3R_OK;
}

// queues the copies of the per-frame voxel COUNTS (h_offs[1..n]), the flag word (h_offs[n+1]), the largest scratch cursor
// (h_offs[n+2]) and the guard's actual verdicts (n bytes from h_offs[n+3])
int tv_read_back(o3r_ctx* ctx, int n) {
    const TvMisc M = tv_misc(ctx, n);
    CU(cudaMemcpyAsync(ctx->last.h_offs + 1, M.fvox, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(ctx->last.h_offs + n + 1, M.flags, 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(ctx->last.h_offs + n + 2, M.max_cursor, 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(ctx->last.h_offs + n + 3, M.actual, (size_t)n, cudaMemcpyDeviceToHost, ctx->st));
    return O3R_OK;
}

// on the landed read-back (and the partial count in h_counters[CNT_PART]).  A raised flag reruns the batch with what the device
// found out; when no window is wide enough, this batch and the context's later ones go to the next engine.
Verdict tv_verdict(o3r_ctx* ctx, TvPlan& pl, int n) {
    const uint32_t* h = ctx->last.h_offs;
    const uint32_t fl = h[n + 1];
    const uint8_t* actual = reinterpret_cast<const uint8_t*>(h + n + 3);
    if (fl) {
        if (trace_on()) fprintf(stderr, "[o3r trace] tile engine flags %u (R %d)\n", fl, pl.R);
        if (fl & TV_FLAG_SPACE) {   // a record list was too short: what the batch needs is known now (+ 25 %)
            ctx->tv.scratch_cap = std::max(ctx->tv.scratch_cap, (size_t)h[n + 2] + h[n + 2] / 4 + 1024);
            ctx->tv.part_cap = std::max(ctx->tv.part_cap, (size_t)ctx->h_counters[CNT_PART] + ctx->h_counters[CNT_PART] / 4 + 1024);
        }
        if (fl & TV_FLAG_PASS) pl.guess.assign(actual, actual + n);   // the bboxes are exact: so is this
        else if (fl & TV_FLAG_RANGE) {   // a disparity beyond the window's reach: widen it
            if (pl.R >= kTvMaxR) { ctx->tv.off = true; return Verdict::NEXT_ENGINE; }
            ctx->tv.R = pl.R + 1;
        }
        return Verdict::RERUN;
    }
    ctx->tv.guess = actual[n - 1];
    // A combined grid fine against the sideways scatter of the points leaves one record per 1-3 points: a 40-byte record per
    // 16-byte point is then a loss, and the sort engine's direct merge of the points serves the context from here on.
    size_t total_vox = 0;
    for (int i = 0; i < n; ++i) total_vox += h[i + 1];
    if ((size_t)ctx->h_counters[CNT_PART] * 4 > total_vox && total_vox > 0) ctx->tv.off = ctx->bk.off = true;
    return Verdict::ACCEPT;
}

}  // namespace
