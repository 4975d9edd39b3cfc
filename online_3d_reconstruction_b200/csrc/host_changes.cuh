// host_changes.cuh — change tracking of the resident cloud (o3r_cloud_track_changes / o3r_cloud_changes[_dev]): the pending
// set D grows by every merged cycle's cells (chg_cycle, called at the end of acc_apply_cycle) and is emitted and emptied by
// the consumer's reads (chg_compute, then chg_reset).  Kernels: changes.cuh.
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "changes.cuh"
#include "host_comm.cuh"

namespace {

// Reserves D's next buffer and the union's scratch for a cycle of up to n_cyc_ub cells, before any launch of the merge:
// an allocation failure then fails the call with the cloud unchanged.  Nothing to do while tracking is off or everything
// is pending.
int chg_reserve(o3r_ctx* ctx, size_t n_cyc_ub) {
    if (!ctx->chg || ctx->chg->all) return O3R_OK;
    ctx->chg->ub = std::min(ctx->chg->ub, ctx->res.n_ub);   // D is a subset of the resident cells
    const size_t in_ub = ctx->chg->ub + n_cyc_ub;
    const uint32_t tiles = cdiv(in_ub, kTileV);
    DevBuf& nxt = ctx->chg->keys[ctx->chg->cur ^ 1];
    if (nxt.cap < in_ub * 8) CU(nxt.ensure(std::max<size_t>(2 * in_ub, (size_t)1 << 20) * 8));   // big steps, as the shard
    CU(ctx->chg->cnt.ensure((size_t)tiles * 4));
    CU(ctx->chg->off.ensure((size_t)tiles * 4));
    CU(ctx->chg->part.ensure(((size_t)tiles + 1) * 4));
    return O3R_OK;
}

// D <- D u ckey[0 .. counters[CNT_CYC]) (the cycle just merged).  Four launches, no device fill, nothing read back.
int chg_cycle(o3r_ctx* ctx, size_t n_cyc_ub) {
    if (!ctx->chg) return O3R_OK;
    ctx->chg->valid = false;
    if (ctx->chg->all) return O3R_OK;   // everything is pending already
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const int cur = ctx->chg->cur, nxt = cur ^ 1;
    const size_t in_ub = ctx->chg->ub + n_cyc_ub;
    const uint32_t tiles = cdiv(in_ub, kTileV);
    const uint64_t* a = ctx->chg->keys[cur].as<uint64_t>();
    const uint64_t* b = ctx->ckey.as<uint64_t>();
    const uint32_t* na = ctx->chg->ub ? cnt + CNT_CHG0 + cur : cnt + CNT_ZERO;
    uint32_t* part = ctx->chg->part.as<uint32_t>();
    LAUNCH(k_chg_part, cdiv((size_t)tiles + 1, kThreads), kThreads, 0, a, na, b, cnt + CNT_CYC, tiles, part);
    LAUNCH_N("k_chg_union_cnt", k_chg_union<false>, tiles, kThreads, 0, a, na, b, cnt + CNT_CYC, part,
             ctx->chg->cnt.as<uint32_t>(), nullptr, nullptr);
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->chg->cnt.as<uint32_t>(), ctx->chg->off.as<uint32_t>(), tiles, cnt + CNT_CHG0 + nxt);
    LAUNCH_N("k_chg_union", k_chg_union<true>, tiles, kThreads, 0, a, na, b, cnt + CNT_CYC, part, nullptr,
             ctx->chg->off.as<uint32_t>(), ctx->chg->keys[nxt].as<uint64_t>());
    ctx->chg->cur = nxt;
    ctx->chg->ub = std::min(in_ub, ctx->res.n_ub);
    return O3R_OK;
}

// Empties the pending set (tracking stays as it is).  No device write: an empty D is known on the host (ub == 0), and
// while it is, the union reads its length from the constant zero slot instead of D's count.
void chg_reset(o3r_ctx* ctx, bool all) {
    ctx->chg->all = all;
    ctx->chg->valid = false;
    ctx->chg->ub = 0;
}

int chg_check_mode(o3r_ctx* ctx) {
    if (ctx->retain())
        return ctx->fail(O3R_ERR_UNSUPPORTED, "change tracking needs an accumulate merge mode (not O3R_MERGE_RETAIN or dont_downsample)");
    return O3R_OK;
}

// The records of the pending cells (every resident cell while everything is pending) with count >= min_points, into
// out / okeys / ocnt, and their number in m.  Kept until the tracked state changes (valid).
int chg_compute(o3r_ctx* ctx) {
    { int rc = chg_check_mode(ctx); if (rc) return rc; }
    if (!ctx->chg) return ctx->fail(O3R_ERR_INVALID, "change tracking is off (o3r_cloud_track_changes)");
    if (ctx->chg->valid) return O3R_OK;
    { int rc = refresh_nres(ctx, false); if (rc) return rc; }
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const ResCells R = res_cells(ctx);
    const bool all = ctx->chg->all;
    const size_t n_ub = all ? ctx->res.n_ub : ctx->chg->ub;   // (ub == 0: D is empty, its count slot is stale)
    ZERO(cnt + CNT_CHGOUT, 8);   // (and CNT_CHGERR)
    if (n_ub) {
        const uint32_t tiles = cdiv(n_ub, kTileV);
        CU(ctx->new_cnt.ensure((size_t)tiles * 4));
        CU(ctx->new_off.ensure((size_t)tiles * 4));
        CU(ctx->chg->pos.ensure(n_ub * 4));
        CU(ctx->chg->out.ensure(n_ub * 16));
        CU(ctx->chg->okeys.ensure(n_ub * 8));
        CU(ctx->chg->ocnt.ensure(n_ub * 4));
        const uint32_t* n_ptr = all ? cnt + CNT_NRES : cnt + CNT_CHG0 + ctx->chg->cur;
        LAUNCH(k_chg_emit_cnt, tiles, kThreads, 0, all ? nullptr : ctx->chg->keys[ctx->chg->cur].as<uint64_t>(), n_ptr,
               R.keys, cnt + CNT_NRES, R.acc, ctx->p.min_points_per_voxel,
               ctx->chg->pos.as<uint32_t>(), ctx->new_cnt.as<uint32_t>(), cnt + CNT_CHGERR);
        LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->new_cnt.as<uint32_t>(), ctx->new_off.as<uint32_t>(), tiles, cnt + CNT_CHGOUT);
        LAUNCH(k_chg_emit, tiles, kThreads, 0, n_ptr, ctx->chg->pos.as<uint32_t>(), R.keys, R.acc, R.rgb, ctx->new_off.as<uint32_t>(),
               ctx->chg->out.as<float4>(), ctx->chg->okeys.as<uint64_t>(), ctx->chg->ocnt.as<uint32_t>());
    }
    { int rc = res_read_back(ctx); if (rc) return rc; }
    const uint32_t* h = ctx->h_counters;
    if (h[CNT_CHGERR]) return ctx->fail(O3R_ERR_INVALID, "internal error: a pending changed cell is not in the resident cloud");
    // (the flag is not cleared and x.pending_check stays set: the next o3r_cloud_downsample still reports the overflow)
    if (ctx->comm && h[CNT_XFLAG]) return x_overflow(ctx);
    if (!all && ctx->chg->ub) ctx->chg->ub = h[CNT_CHG0 + ctx->chg->cur];
    ctx->chg->m = h[CNT_CHGOUT];
    ctx->chg->valid = true;
    return O3R_OK;
}

}  // namespace
