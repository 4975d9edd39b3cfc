// host_sort.cuh — drivers of the segmented radix sort and of engine 1 (VoxelGrid on sorted leaf indices)
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "host_ctx.cuh"

namespace {

// ---- radix sort driver -----------------------------------------------------------------------------------------
// The caller provides ghist [n_seg][passes][256] (already filled) and plan.
// Segments that can reach kRsWideSeg items publish their look-back prefixes in 64-bit status words: a digit's inclusive
// prefix would overflow the 30 count bits of the 32-bit word.
template <typename KeyT, typename StT>
int sort_pairs_t(o3r_ctx* ctx, KeyT* k0, KeyT* k1, uint32_t* v0, uint32_t* v1, const uint32_t* seg_off, int n_seg,
                 size_t per_seg_cap, const SortPlan* plan, int passes, int iota_first, const uint32_t* ghist,
                 int ghist_is_prefix) {
    const uint32_t tiles_ub = std::max(1u, cdiv(per_seg_cap, kRsTile));
    const size_t st_words = (size_t)n_seg * tiles_ub * kRsBins;
    // status words for every pass + one ticket per pass, cleared with one memset
    const size_t bytes = st_words * passes * sizeof(StT) + 64 * 4;
    CU(ctx->hist.ensure(bytes));
    ZERO(ctx->hist.p, bytes);
    StT* status = ctx->hist.as<StT>();
    uint32_t* tickets = reinterpret_cast<uint32_t*>(status + st_words * passes);
    const uint32_t grid = tiles_ub * (uint32_t)n_seg;
    const char* name = sizeof(StT) == 4 ? (sizeof(KeyT) == 4 ? "k_rs_onesweep_u32" : "k_rs_onesweep_u64")
                                        : (sizeof(KeyT) == 4 ? "k_rs_onesweep_u32_wide" : "k_rs_onesweep_u64_wide");
    for (int p = 0; p < passes; ++p)
        LAUNCH_N(name, (k_rs_onesweep<KeyT, StT>), grid, kThreads, rs_scatter_smem<KeyT>(), k0, k1, v0, v1, seg_off, plan,
                 p, tiles_ub, ghist, status + st_words * p, tickets + p, iota_first, ghist_is_prefix);
    return O3R_OK;
}

template <typename KeyT>
int sort_pairs(o3r_ctx* ctx, KeyT* k0, KeyT* k1, uint32_t* v0, uint32_t* v1, const uint32_t* seg_off, int n_seg,
               size_t per_seg_cap, const SortPlan* plan, int passes, int iota_first, const uint32_t* ghist,
               int ghist_is_prefix = 1) {
    if (per_seg_cap >= kRsWideSeg)
        return sort_pairs_t<KeyT, uint64_t>(ctx, k0, k1, v0, v1, seg_off, n_seg, per_seg_cap, plan, passes, iota_first, ghist,
                                            ghist_is_prefix);
    return sort_pairs_t<KeyT, uint32_t>(ctx, k0, k1, v0, v1, seg_off, n_seg, per_seg_cap, plan, passes, iota_first, ghist,
                                        ghist_is_prefix);
}

// ---- engine 1: VoxelGrid on segments whose leaf indices already sit in sortbuf keys0 ----------------------------
struct SortU32 { uint32_t *k0, *k1, *v0, *v1; };

int carve_sort_u32(o3r_ctx* ctx, size_t n, SortU32& s) {
    const size_t n4 = (n + 63) & ~(size_t)63;
    CU(ctx->sortbuf.ensure(n4 * 16));
    s.k0 = ctx->sortbuf.as<uint32_t>();
    s.k1 = s.k0 + n4; s.v0 = s.k1 + n4; s.v1 = s.v0 + n4;
    return O3R_OK;
}

// digit layout, whole-segment histograms and pass plan of a segmented u32 sort whose keys sit in sb.k0
// (grids[s].key_bits = live key bits of segment s); leaves the plan in ctx->plan_all, the histograms in ctx->ghist
int sort_segments_plan(o3r_ctx* ctx, const SortU32& sb, const uint32_t* seg_off, int n_seg, size_t per_seg_cap,
                       const GridParams* grids) {
    const size_t gh_bytes = (size_t)n_seg * kMaxPasses * kRsBins * 4;
    CU(ctx->ghist.ensure(gh_bytes));
    CU(ctx->plan_all.ensure((size_t)n_seg * sizeof(SortPlan)));
    ZERO(ctx->ghist.p, gh_bytes);
    SortPlan* plan = ctx->plan_all.as<SortPlan>();
    // digit layout from each segment's live index bits (<= 31 -> at most 4 passes)
    LAUNCH(k_rs_layout, cdiv(n_seg, 64), 64, 0, n_seg, grids, 31, plan);
    LAUNCH_N("k_rs_ghist_u32", (k_rs_ghist<uint32_t, 4>), dim3(std::max(1u, cdiv(per_seg_cap, kRsTile)), n_seg),
             kThreads, 0, sb.k0, seg_off, plan, ctx->ghist.as<uint32_t>());
    LAUNCH(k_rs_plan, n_seg, kThreads, 0, ctx->ghist.as<uint32_t>(), seg_off, plan, grids);
    return O3R_OK;
}

// sorts + reduces; out/out_off sized by the caller.  CNT_VOX receives the total.  track_cells / out_base only serve the
// unfiltered reduction (min_points <= 1, no keys / counts).
int vg_sorted_reduce(o3r_ctx* ctx, const SortU32& sb, const float4* pts, const uint32_t* seg_off, int n_seg,
                     size_t per_seg_cap, const GridParams* grids, float ix, float iy, float iz, uint32_t min_points,
                     int z_shift, float4* out, uint32_t* out_off, uint64_t* out_keys, uint32_t* out_counts,
                     bool track_cells = false, const uint32_t* out_base = nullptr) {
    int rcs = sort_segments_plan(ctx, sb, seg_off, n_seg, per_seg_cap, grids);
    if (rcs) return rcs;
    SortPlan* plan = ctx->plan_all.as<SortPlan>();
    int rc = sort_pairs<uint32_t>(ctx, sb.k0, sb.k1, sb.v0, sb.v1, seg_off, n_seg, per_seg_cap, plan, 4, 1,
                                  ctx->ghist.as<uint32_t>());
    if (rc) return rc;
    VgArgs A;
    A.keys0 = sb.k0; A.keys1 = sb.k1; A.vals0 = sb.v0; A.vals1 = sb.v1;
    A.seg_off = seg_off; A.plan = plan; A.grids = grids; A.pts = pts;
    A.tiles_ub = std::max(1u, cdiv(per_seg_cap, kTileV));
    A.min_points = min_points; A.z_shift = z_shift;
    A.lx_inv = ix; A.ly_inv = iy; A.lz_inv = iz;
    const size_t nt = (size_t)A.tiles_ub * n_seg;
    CU(ctx->head_cnt.ensure(nt * 4));
    CU(ctx->head_off.ensure(nt * 4));
    const dim3 grid(A.tiles_ub, n_seg);
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    LAUNCH(k_vg_heads, grid, kThreads, 0, A, ctx->head_cnt.as<uint32_t>());
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->head_cnt.as<uint32_t>(), ctx->head_off.as<uint32_t>(), (uint32_t)nt,
           cnt + CNT_VOX);
    const size_t wbytes = 64 + (nt + 1) * sizeof(RunCarry);
    CU(ctx->runwork.ensure(wbytes));
    ZERO(ctx->runwork.p, wbytes);
    const bool full = min_points > 1 || out_keys || out_counts;
    LAUNCH_N(full ? "k_vg_reduce_w_full" : "k_vg_reduce_w", (full ? k_vg_reduce_w<true> : k_vg_reduce_w<false>),
             (uint32_t)nt, kThreads, 0, A, ctx->head_off.as<uint32_t>(), cnt + CNT_VOX, out, out_off, n_seg,
             ctx->runwork.as<uint32_t>(), reinterpret_cast<RunCarry*>(ctx->runwork.as<char>() + 64), track_cells ? 1 : 0,
             ctx->inv_c, ctx->inv_cz, reinterpret_cast<int*>(cnt + CNT_CELLBB), out_base, out_keys, out_counts);
    return O3R_OK;
}

// engine 1 over the one segment [0, n) of pts, whose bounds are already in `seg` and whose grid is in ctx->grids: leaf
// indices, sort, reduction into `out` (and `out_keys` / `out_counts` when given).  Waits for the stream; *m = records.
int vg_one_segment(o3r_ctx* ctx, const float4* pts, const uint32_t* seg, size_t n, float ix, float iy, float iz,
                   uint32_t min_points, int z_shift, float4* out, uint64_t* out_keys, uint32_t* out_counts, size_t* m) {
    CU(ctx->vox_off.ensure(2 * 4));
    SortU32 sb;
    int rc = carve_sort_u32(ctx, n, sb);
    if (rc) return rc;
    const GridParams* grids = ctx->grids.as<GridParams>();
    LAUNCH(k_vg_key, dim3(std::min<uint32_t>(cdiv(n, kThreads), 148 * 16), 1), kThreads, 0, pts, seg, grids, z_shift, sb.k0);
    rc = vg_sorted_reduce(ctx, sb, pts, seg, 1, n, grids, ix, iy, iz, min_points, z_shift, out, ctx->vox_off.as<uint32_t>(),
                          out_keys, out_counts);
    if (rc) return rc;
    rc = read_counters(ctx);
    if (rc) return rc;
    *m = ctx->h_counters[CNT_VOX];
    return O3R_OK;
}

}  // namespace
