// host_sor.cuh — StatisticalOutlierRemoval on the frames of a chunk
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "host_sort.cuh"

namespace {

// ---- pcl::StatisticalOutlierRemoval on the frames of a chunk (pose_functions.cpp:1673-1686) -----------------------------
// in: pts with segment offsets seg_off[n_seg + 1] (device).  out: ctx->sor.pts / ctx->sor.off (same layout, kept points
// in their original order).  Uses the sort buffers (free again afterwards) and ctx->bbox / ctx->sor.spts as scratch.
int sor_filter(o3r_ctx* ctx, const SortU32& sb, const float4* pts, const uint32_t* seg_off, int n_seg, size_t per_seg_cap,
               int mean_k, double stddev_mul) {
    if (mean_k < 1) return ctx->fail(O3R_ERR_INVALID, "sor_mean_k must be positive");
    if (mean_k + 1 > kSorMaxK) return ctx->fail(O3R_ERR_INVALID, "sor_mean_k too large (max 127)");
    const size_t cap = per_seg_cap * n_seg;
    const uint32_t tiles = std::max(1u, cdiv(per_seg_cap, kTileV));
    CU(ctx->sor.pts.ensure(cap * 16));
    CU(ctx->sor.off.ensure((size_t)(n_seg + 1) * 4));
    CU(ctx->sor.dist.ensure(cap * 4));
    CU(ctx->sor.skeys.ensure(cap * 4));
    CU(ctx->sor.svals.ensure(cap * 4));
    CU(ctx->sor.spts.ensure(cap * 16));
    CU(ctx->sor.grids.ensure((size_t)n_seg * sizeof(SorGrid)));
    CU(ctx->sor.pgrids.ensure((size_t)n_seg * sizeof(GridParams)));
    CU(ctx->sor.rows.ensure((size_t)n_seg * (kSorCellsCap + 1) * 4));
    CU(ctx->sor.thr.ensure((size_t)n_seg * 8));
    CU(ctx->sor.cnt.ensure((size_t)tiles * n_seg * 4));
    CU(ctx->sor.cntoff.ensure((size_t)tiles * n_seg * 4));
    CU(ctx->bbox.ensure((size_t)n_seg * 6 * 4));
    SorGrid* grids = ctx->sor.grids.as<SorGrid>();
    GridParams* pgrids = ctx->sor.pgrids.as<GridParams>();
    uint32_t* cell_start = ctx->sor.rows.as<uint32_t>();   // [n_seg][kSorCellsCap + 1]
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const uint32_t gl = std::min<uint32_t>(std::max(1u, cdiv(per_seg_cap, kThreads)), 148 * 4);
    FILL(ctx->bbox.as<uint32_t>(), (size_t)(n_seg) * 24, FILL_BBOX);
    LAUNCH(k_bbox_pts, dim3(tiles, n_seg), kThreads, 0, pts, seg_off, 0, ctx->bbox.as<uint32_t>());
    LAUNCH(k_sor_grid, cdiv(n_seg, 64), 64, 0, n_seg, ctx->bbox.as<uint32_t>(), seg_off, mean_k, grids, pgrids);
    const size_t heap_bytes = (size_t)(mean_k + 1) * kSorThreads * 4;
    CU(cudaFuncSetAttribute(k_sor_knn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)heap_bytes));
    CU(cudaFuncSetAttribute(k_sor_calib, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)heap_bytes));
    SortPlan* plan = ctx->plan_all.as<SortPlan>();
    // grid build, twice: on the density guess, then on the cell the calibration derives from 128 exact sample queries per frame
    for (int round = 0; round < 2; ++round) {
        LAUNCH(k_sor_key, dim3(gl, n_seg), kThreads, 0, pts, seg_off, grids, sb.k0);
        int rc = sort_segments_plan(ctx, sb, seg_off, n_seg, per_seg_cap, pgrids);
        if (rc) return rc;
        plan = ctx->plan_all.as<SortPlan>();
        rc = sort_pairs<uint32_t>(ctx, sb.k0, sb.k1, sb.v0, sb.v1, seg_off, n_seg, per_seg_cap, plan, 4, 1, ctx->ghist.as<uint32_t>());
        if (rc) return rc;
        LAUNCH(k_sor_cells, dim3(gl, n_seg), kThreads, 0, sb.k0, sb.k1, sb.v0, sb.v1, plan, pts, seg_off, grids, cell_start,
               ctx->sor.skeys.as<uint32_t>(), ctx->sor.svals.as<uint32_t>(), ctx->sor.spts.as<float4>());
        if (round == 0)
            LAUNCH(k_sor_calib, n_seg, kSorThreads, heap_bytes, ctx->sor.spts.as<float4>(), ctx->sor.skeys.as<uint32_t>(), seg_off, grids,
                   pgrids, ctx->bbox.as<uint32_t>(), cell_start, mean_k);
    }
    CU(ctx->sor.hard.ensure(cap * 8 + 64));
    uint32_t* n_hard = reinterpret_cast<uint32_t*>(ctx->sor.hard.as<char>() + cap * 8);
    ZERO(n_hard, 4);
    CU(cudaFuncSetAttribute(k_sor_knn_hard, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)heap_bytes));
    LAUNCH(k_sor_knn, dim3(std::max(1u, cdiv(per_seg_cap, kSorThreads)), n_seg), kSorThreads, heap_bytes, ctx->sor.spts.as<float4>(),
           ctx->sor.skeys.as<uint32_t>(), ctx->sor.svals.as<uint32_t>(), seg_off, grids, cell_start, mean_k,
           ctx->sor.dist.as<float>(), ctx->sor.hard.as<uint2>(), n_hard);
    LAUNCH(k_sor_knn_hard, std::max(1u, cdiv(cap, kSorThreads)), kSorThreads, heap_bytes, ctx->sor.spts.as<float4>(),
           ctx->sor.skeys.as<uint32_t>(), ctx->sor.svals.as<uint32_t>(), seg_off, grids, cell_start, mean_k,
           ctx->sor.dist.as<float>(), ctx->sor.hard.as<uint2>(), n_hard);
    LAUNCH(k_sor_stats, n_seg, kThreads, 0, ctx->sor.dist.as<float>(), seg_off, stddev_mul, ctx->sor.thr.as<double>());
    LAUNCH(k_sor_count, dim3(tiles, n_seg), kThreads, 0, ctx->sor.dist.as<float>(), seg_off, ctx->sor.thr.as<double>(), tiles,
           ctx->sor.cnt.as<uint32_t>());
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->sor.cnt.as<uint32_t>(), ctx->sor.cntoff.as<uint32_t>(), (uint32_t)((size_t)tiles * n_seg),
           cnt + CNT_PTS);
    LAUNCH(k_sor_compact, dim3(tiles, n_seg), kThreads, 0, pts, ctx->sor.dist.as<float>(), seg_off, ctx->sor.thr.as<double>(), tiles,
           ctx->sor.cntoff.as<uint32_t>(), cnt + CNT_PTS, n_seg, ctx->sor.pts.as<float4>(), ctx->sor.off.as<uint32_t>());
    return O3R_OK;
}

}  // namespace
