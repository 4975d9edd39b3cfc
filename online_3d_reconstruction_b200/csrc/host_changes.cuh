// host_changes.cuh — change tracking of the resident cloud (o3r_cloud_track_changes / o3r_cloud_changes[_dev]): the pending
// set D grows by every merged cycle's cells (chg_cycle, called at the end of acc_apply_cycle) and is emitted and emptied by
// the consumer's reads (chg_compute, then chg_reset).  Kernels: changes.cuh.
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "changes.cuh"
#include "host_merge.cuh"

namespace {

// Reserves D's next buffer and the union's scratch for a cycle of up to n_cyc_ub cells, before any launch of the merge:
// an allocation failure then fails the call with the cloud unchanged.  Nothing to do while tracking is off or everything
// is pending.
int chg_reserve(o3r_ctx* ctx, size_t n_cyc_ub) {
    if (!ctx->chg_on || ctx->chg_all) return O3R_OK;
    ctx->chg_ub = std::min(ctx->chg_ub, ctx->n_res_ub);   // D is a subset of the resident cells
    const size_t in_ub = ctx->chg_ub + n_cyc_ub;
    const uint32_t tiles = cdiv(in_ub, kTileV);
    DevBuf& nxt = ctx->chg_keys[ctx->chg_cur ^ 1];
    if (nxt.cap < in_ub * 8) CU(nxt.ensure(std::max<size_t>(2 * in_ub, (size_t)1 << 20) * 8));   // big steps, as the shard
    CU(ctx->chg_cnt.ensure((size_t)tiles * 4));
    CU(ctx->chg_off.ensure((size_t)tiles * 4));
    CU(ctx->chg_part.ensure(((size_t)tiles + 1) * 4));
    return O3R_OK;
}

// D <- D u ckey[0 .. counters[CNT_CYC]) (the cycle just merged).  Four launches, no device fill, nothing read back.
int chg_cycle(o3r_ctx* ctx, size_t n_cyc_ub) {
    if (!ctx->chg_on) return O3R_OK;
    ctx->chg_valid = false;
    if (ctx->chg_all) return O3R_OK;   // everything is pending already
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const int cur = ctx->chg_cur, nxt = cur ^ 1;
    const size_t in_ub = ctx->chg_ub + n_cyc_ub;
    const uint32_t tiles = cdiv(in_ub, kTileV);
    const uint64_t* a = ctx->chg_keys[cur].as<uint64_t>();
    const uint64_t* b = ctx->ckey.as<uint64_t>();
    const uint32_t* na = ctx->chg_ub ? cnt + CNT_CHG0 + cur : cnt + CNT_ZERO;
    uint32_t* part = ctx->chg_part.as<uint32_t>();
    LAUNCH(k_chg_part, cdiv((size_t)tiles + 1, kThreads), kThreads, 0, a, na, b, cnt + CNT_CYC, tiles, part);
    LAUNCH_N("k_chg_union_cnt", k_chg_union<false>, tiles, kThreads, 0, a, na, b, cnt + CNT_CYC, part,
             ctx->chg_cnt.as<uint32_t>(), nullptr, nullptr);
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->chg_cnt.as<uint32_t>(), ctx->chg_off.as<uint32_t>(), tiles, cnt + CNT_CHG0 + nxt);
    LAUNCH_N("k_chg_union", k_chg_union<true>, tiles, kThreads, 0, a, na, b, cnt + CNT_CYC, part, nullptr,
             ctx->chg_off.as<uint32_t>(), ctx->chg_keys[nxt].as<uint64_t>());
    ctx->chg_cur = nxt;
    ctx->chg_ub = std::min(in_ub, ctx->n_res_ub);
    return O3R_OK;
}

// Empties the pending set (tracking stays as it is).  No device write: an empty D is known on the host (chg_ub == 0), and
// while it is, the union reads its length from the constant zero slot instead of D's count.
void chg_reset(o3r_ctx* ctx, bool all) {
    ctx->chg_all = all;
    ctx->chg_valid = false;
    ctx->chg_ub = 0;
}

int chg_check_mode(o3r_ctx* ctx) {
    if (ctx->retain())
        return ctx->fail(O3R_ERR_UNSUPPORTED, "change tracking needs an accumulate merge mode (not O3R_MERGE_RETAIN or dont_downsample)");
    return O3R_OK;
}

// The records of the pending cells (every resident cell while everything is pending) with count >= min_points, into
// chg_out / chg_okeys / chg_ocnt, and their number in chg_m.  Kept until the tracked state changes (chg_valid).
int chg_compute(o3r_ctx* ctx) {
    { int rc = chg_check_mode(ctx); if (rc) return rc; }
    if (!ctx->chg_on) return ctx->fail(O3R_ERR_INVALID, "change tracking is off (o3r_cloud_track_changes)");
    if (ctx->chg_valid) return O3R_OK;
    { int rc = refresh_nres(ctx, false); if (rc) return rc; }
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const int cur = ctx->res_cur;
    const bool all = ctx->chg_all;
    const size_t n_ub = all ? ctx->n_res_ub : ctx->chg_ub;   // (chg_ub == 0: D is empty, its count slot is stale)
    ZERO(cnt + CNT_CHGOUT, 8);   // (and CNT_CHGERR)
    if (n_ub) {
        const uint32_t tiles = cdiv(n_ub, kTileV);
        CU(ctx->new_cnt.ensure((size_t)tiles * 4));
        CU(ctx->new_off.ensure((size_t)tiles * 4));
        CU(ctx->chg_pos.ensure(n_ub * 4));
        CU(ctx->chg_out.ensure(n_ub * 16));
        CU(ctx->chg_okeys.ensure(n_ub * 8));
        CU(ctx->chg_ocnt.ensure(n_ub * 4));
        const uint32_t* n_ptr = all ? cnt + CNT_NRES : cnt + CNT_CHG0 + ctx->chg_cur;
        LAUNCH(k_chg_emit_cnt, tiles, kThreads, 0, all ? nullptr : ctx->chg_keys[ctx->chg_cur].as<uint64_t>(), n_ptr,
               ctx->res_keys[cur].as<uint64_t>(), cnt + CNT_NRES, ctx->res_acc[cur].as<float4>(), ctx->p.min_points_per_voxel,
               ctx->chg_pos.as<uint32_t>(), ctx->new_cnt.as<uint32_t>(), cnt + CNT_CHGERR);
        LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->new_cnt.as<uint32_t>(), ctx->new_off.as<uint32_t>(), tiles, cnt + CNT_CHGOUT);
        LAUNCH(k_chg_emit, tiles, kThreads, 0, n_ptr, ctx->chg_pos.as<uint32_t>(), ctx->res_keys[cur].as<uint64_t>(),
               ctx->res_acc[cur].as<float4>(), ctx->res_rgb[cur].as<uint4>(), ctx->new_off.as<uint32_t>(),
               ctx->chg_out.as<float4>(), ctx->chg_okeys.as<uint64_t>(), ctx->chg_ocnt.as<uint32_t>());
    }
    { int rc = read_counters(ctx); if (rc) return rc; }
    const uint32_t* h = ctx->h_counters;
    ctx->n_res_ub = h[CNT_NRES];
    ctx->n_res_exact = true;
    if (h[CNT_CHGERR]) return ctx->fail(O3R_ERR_INVALID, "internal error: a pending changed cell is not in the resident cloud");
    // (the flag is not cleared and x_pending_check stays set: the next o3r_cloud_downsample still reports the overflow)
    if (ctx->comm && h[CNT_XFLAG])
        return ctx->fail(O3R_ERR_CAPACITY, "exchange slot overflow: cells were dropped; create the communicator with more slot_cells");
    if (!all && ctx->chg_ub) ctx->chg_ub = h[CNT_CHG0 + ctx->chg_cur];
    ctx->chg_m = h[CNT_CHGOUT];
    ctx->chg_valid = true;
    return O3R_OK;
}

}  // namespace
