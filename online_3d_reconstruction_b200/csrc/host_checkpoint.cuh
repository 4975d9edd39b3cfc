// host_checkpoint.cuh — checkpoints of the resident map (o3r_cloud_export_cells / o3r_cloud_import_cells /
// o3r_cloud_export_points).  An export packs the accumulators into o3r_cell records (k_cells_pack) and copies them out; an
// import stages the caller's records in a buffer of its own (ck_cells), validates every record on the device (k_cells_check)
// and only then merges them as one cycle through the ordinary engine-2 merge.  Kernels: checkpoint.cuh.
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "checkpoint.cuh"
#include "host_comm.cuh"

namespace {

int ck_check_cells_mode(o3r_ctx* ctx) {
    if (ctx->retain())
        return ctx->fail(O3R_ERR_UNSUPPORTED, "cell checkpoints need an accumulate merge mode (not O3R_MERGE_RETAIN or dont_downsample): "
                                              "use o3r_cloud_export_points");
    return O3R_OK;
}

int export_cells_impl(o3r_ctx* ctx, o3r_cell* out, size_t cap, size_t* n_out) {
    { int rc = ck_check_cells_mode(ctx); if (rc) return rc; }
    { int rc = refresh_nres(ctx, false); if (rc) return rc; }
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const size_t n_ub = ctx->res.n_ub;
    // pack and queue the copy behind it unless the buffer is known to be short; one sync for the copy and the exact count
    const bool fill = out && cap && n_ub && !res_exceeds(ctx, cap);
    if (fill) {
        CU(ctx->ck_cells.ensure(n_ub * sizeof(o3r_cell)));
        const ResCells R = res_cells(ctx);
        LAUNCH(k_cells_pack, std::min<uint32_t>(cdiv(n_ub, kThreads), 148 * 16), kThreads, 0, cnt + CNT_NRES, R.keys, R.acc,
               R.rgb, ctx->ck_cells.as<o3r_cell>());
        CU(cudaMemcpyAsync(out, ctx->ck_cells.p, std::min(cap, n_ub) * sizeof(o3r_cell), cudaMemcpyDeviceToHost, ctx->st));
    }
    { int rc = res_read_back(ctx); if (rc) return rc; }
    const size_t m = ctx->res.n_ub;
    if (ctx->comm && ctx->h_counters[CNT_XFLAG]) return x_overflow(ctx);   // (not cleared: the next o3r_cloud_downsample reports it too)
    *n_out = m;
    if (!out && cap == 0) return O3R_OK;
    if (cap < m) return ctx->fail(O3R_ERR_CAPACITY, "output buffer too small");
    return O3R_OK;
}

std::string ck_reasons(uint32_t f) {
    static const struct { uint32_t bit; const char* what; } kNames[] = {
        {o3r::kCkKeyBit63, "bit 63 of the key is set"},
        {o3r::kCkKeyRange, "a key field is outside +-(2^20 - 1) cells"},
        {o3r::kCkZeroCount, "n == 0"},
        {o3r::kCkNotFinite, "a coordinate sum is not finite"},
        {o3r::kCkColour, "a colour sum exceeds 255 * n"},
        {o3r::kCkPad, "pad != 0"},
        {o3r::kCkOwner, "the cell belongs to another rank (hash64(key) % world != rank)"},
    };
    std::string s;
    for (const auto& r : kNames)
        if (f & r.bit) { if (!s.empty()) s += "; "; s += r.what; }
    return s;
}

int import_cells_impl(o3r_ctx* ctx, const o3r_cell* cells, size_t n) {
    { int rc = ck_check_cells_mode(ctx); if (rc) return rc; }
    if (n == 0) return O3R_OK;
    if (n >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "too many cell records for one import (2^32 or more)");
    CU(ctx->ck_cells.ensure(n * sizeof(o3r_cell)));
    CU(ctx->ck_res.ensure(16));
    CU(cudaMemcpyAsync(ctx->ck_cells.p, cells, n * sizeof(o3r_cell), cudaMemcpyHostToDevice, ctx->st));
    const unsigned long long init[2] = {~0ull, 0ull};
    { int rcu = upload_small(ctx, ctx->ck_res.p, init, sizeof(init)); if (rcu) return rcu; }
    LAUNCH(k_cells_check, std::min<uint32_t>(cdiv(n, kThreads), 148 * 8), kThreads, 0, ctx->ck_cells.as<o3r_cell>(), (uint32_t)n,
           ctx->comm ? (uint32_t)ctx->world : 0u, (uint32_t)ctx->rank, ctx->ck_res.as<unsigned long long>());
    unsigned long long res[2];
    CU(cudaMemcpyAsync(res, ctx->ck_res.p, sizeof(res), cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));   // the caller's records are on the device: it may free them whatever follows
    if (res[1]) {
        char head[96];
        snprintf(head, sizeof(head), "cell record %llu refused: ", res[0] >> 32);
        return ctx->fail(O3R_ERR_INVALID, head + ck_reasons((uint32_t)res[0]) + " (nothing was merged)");
    }
    AccItemsCells items{ctx->ck_cells.as<o3r_cell>(), nullptr, nullptr};
    int rc = acc_build_cycle(ctx, items, n, true, nullptr);
    if (rc) return rc;
    return acc_apply_cycle(ctx);
}

int export_points_impl(o3r_ctx* ctx, o3r_point* out, size_t cap, size_t* n_out) {
    if (!ctx->retain())
        return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_export_points needs O3R_MERGE_RETAIN or dont_downsample: use o3r_cloud_export_cells");
    if (ctx->comm)
        return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_export_points on a sharded point cloud: its frame-order tags cannot be exported");
    return copy_out(ctx, ctx->res.cloud.as<float4>(), ctx->res.n_cloud, out, cap, n_out);
}

}  // namespace
