// host_merge.cuh — engine 2: the incremental merge of a cycle into the resident accumulators
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "host_sort.cuh"

namespace {

int chg_reserve(o3r_ctx* ctx, size_t n_cyc_ub);   // change tracking (host_changes.cuh)
int chg_cycle(o3r_ctx* ctx, size_t n_cyc_ub);

// ---- engine 2: merge `n` items (points or partial cells) into the resident accumulators --------------------------
inline int bits_for(long long range) { int b = 0; while ((1ll << b) <= range) ++b; return b; }

template <typename KeyT, typename Items>
int acc_build_cycle_t(o3r_ctx* ctx, Items items, size_t n, bool use_resident, const KeyCodec& kc, int total_bits,
                      const uint32_t* n_dev = nullptr) {
    const int passes = std::max(1, (total_bits + kRsMaxBits - 1) / kRsMaxBits);
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const size_t n4 = (n + 63) & ~(size_t)63;
    Tr tr("acc_build");
    CU(ctx->sortbuf.ensure(n4 * (2 * sizeof(KeyT) + 8)));
    tr.mark("sortbuf.ensure");
    KeyT* k0 = ctx->sortbuf.as<KeyT>();
    KeyT* k1 = k0 + n4;
    uint32_t* v0 = reinterpret_cast<uint32_t*>(k1 + n4);
    uint32_t* v1 = v0 + n4;
    CU(ctx->seg2.ensure(16));
    CU(ctx->ghist.ensure(kMaxPasses * kRsBins * 4));
    CU(ctx->plan_v2.ensure(sizeof(SortPlan)));
    if (!n_dev) {
        const uint32_t seg_h[2] = {0u, (uint32_t)n};
        int rcu = upload_small(ctx, ctx->seg2.p, seg_h, 8);
        if (rcu) return rcu;
    }   // (else k_acc_key writes the segment from the device-side count)
    ZERO(ctx->ghist.p, kMaxPasses * kRsBins * 4);
    ZERO(cnt + CNT_NEW, 4);
    const uint32_t* seg = ctx->seg2.as<uint32_t>();
    const uint32_t gk = std::min<uint32_t>(cdiv(n, kThreads), 148 * 8);
    SortPlan* plan = ctx->plan_v2.as<SortPlan>();
    LAUNCH(k_rs_layout, 1, 32, 0, 1, (const GridParams*)nullptr, total_bits, plan);
    LAUNCH_N("k_acc_key", (k_acc_key<KeyT, Items>), gk, kThreads, 0, items, (uint32_t)n, ctx->inv_c, ctx->inv_cz, kc, plan,
             k0, v0, ctx->ghist.as<uint32_t>(), n_dev, ctx->seg2.as<uint32_t>());
    LAUNCH(k_rs_plan, 1, kThreads, 0, ctx->ghist.as<uint32_t>(), seg, plan, (const GridParams*)nullptr);
    tr.mark("key+plan");
    int rc = sort_pairs<KeyT>(ctx, k0, k1, v0, v1, seg, 1, n, plan, passes, 0, ctx->ghist.as<uint32_t>());
    if (rc) return rc;
    tr.mark("sort_pairs");
    AccArgs<KeyT> A;
    A.keys0 = k0; A.keys1 = k1; A.vals0 = v0; A.vals1 = v1;
    A.seg_off = seg; A.plan = plan;
    A.tiles_ub = cdiv(n, kTileV);
    A.kc = kc;
    const int cur = ctx->res_cur;
    A.res_keys = ctx->res_keys[cur].as<uint64_t>();
    A.res_acc = ctx->res_acc[cur].as<float4>();
    A.res_rgb = ctx->res_rgb[cur].as<uint4>();
    A.n_res_ptr = cnt + (use_resident ? CNT_NRES : CNT_ZERO);
    CU(ctx->head_cnt.ensure((size_t)A.tiles_ub * 4));
    CU(ctx->head_off.ensure((size_t)A.tiles_ub * 4));
    // one record per cell of the cycle (<= n_cyc_ub <= n), reserved in big steps so steady-state cycles never reallocate
    const size_t cyc_cap = std::max<size_t>(std::min<size_t>(n, ctx->n_cyc_ub ? ctx->n_cyc_ub : n), (size_t)1 << 20);
    CU(ctx->ckey.ensure(cyc_cap * 8));
    CU(ctx->cacc.ensure(cyc_cap * 16));
    CU(ctx->crgb.ensure(cyc_cap * 16));
    const size_t wbytes = 64 + ((size_t)A.tiles_ub + 1) * sizeof(RunCarry);
    CU(ctx->runwork.ensure(wbytes));
    ZERO(ctx->runwork.p, wbytes);
    tr.mark("ensures");
    LAUNCH_N("k_acc_heads", (k_acc_heads<KeyT>), A.tiles_ub, kThreads, 0, A, v0, v1, ctx->head_cnt.as<uint32_t>(),
             cnt + CNT_NEW);
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->head_cnt.as<uint32_t>(), ctx->head_off.as<uint32_t>(), A.tiles_ub,
           cnt + CNT_CYC);
    LAUNCH_N("k_acc_reduce", (k_acc_reduce<KeyT, Items>), A.tiles_ub, kThreads, 0, A, items, ctx->head_off.as<uint32_t>(),
             ctx->ckey.as<uint64_t>(), ctx->cacc.as<float4>(), ctx->crgb.as<uint4>(), ctx->runwork.as<uint32_t>(),
             reinterpret_cast<RunCarry*>(ctx->runwork.as<char>() + 64));
    tr.mark("heads+reduce");
    return O3R_OK;
}

// Tightens the host's upper bound of the resident cell count from the read-back of the last merge.
int refresh_nres(o3r_ctx* ctx, bool block) {
    if (ctx->n_res_exact) return O3R_OK;
    if (block) CU(cudaEventSynchronize(ctx->ev_nres));
    else if (cudaEventQuery(ctx->ev_nres) != cudaSuccess) { cudaGetLastError(); return O3R_OK; }
    ctx->n_res_ub = *ctx->h_nres;
    ctx->n_res_exact = true;
    return O3R_OK;
}

// Builds the cycle's cell list (ckey/cacc/crgb, count in counters[CNT_CYC]) from items, continuing from the resident sums when
// `use_resident`.  `bb` = {imin,jmin,kmin,imax,jmax,kmax} of the items' combined-grid cells when the caller already
// knows it (host), else null.  Leaves h_counters[CNT_CYC], [CNT_NEW] valid.
template <typename Items>
int acc_build_cycle(o3r_ctx* ctx, const Items& items, size_t n, bool use_resident, const int* bb) {
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    ctx->n_cyc_ub = 0;
    ctx->h_counters[CNT_CYC] = ctx->h_counters[CNT_NEW] = 0;
    if (n == 0) return O3R_OK;
    { int rc = refresh_nres(ctx, false); if (rc) return rc; }
    if (n >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "batch too large for 32-bit indices");
    int hb[6];
    if (!bb) {
        FILL(cnt + CNT_CELLBB, 24, FILL_CELLBB);
        LAUNCH_N("k_acc_cellbb", (k_acc_cellbb<Items>), std::min<uint32_t>(cdiv(n, kThreads), 148 * 8), kThreads, 0, items,
                 (uint32_t)n, ctx->inv_c, ctx->inv_cz, reinterpret_cast<int*>(cnt + CNT_CELLBB));
        int rc = read_counters(ctx);
        if (rc) return rc;
        memcpy(hb, ctx->h_counters + CNT_CELLBB, sizeof(hb));
        bb = hb;
    }
    const int lim = (1 << 20) - 1;
    for (int a = 0; a < 3; ++a)
        if (bb[a] < -lim || bb[3 + a] > lim || bb[3 + a] < bb[a])
            return ctx->fail(O3R_ERR_INVALID, "cloud extends beyond +-2^20 combined-grid cells (or is not finite)");
    KeyCodec kc;
    kc.imin = bb[0]; kc.jmin = bb[1]; kc.kmin = bb[2];
    kc.wi = bits_for((long long)bb[3] - bb[0]);
    kc.wj = bits_for((long long)bb[4] - bb[1]);
    const int total = kc.wi + kc.wj + bits_for((long long)bb[5] - bb[2]);
    // the cycle cannot touch more cells than its cell range holds (nor more than it has items)
    const double range_cells = ((double)bb[3] - bb[0] + 1) * ((double)bb[4] - bb[1] + 1) * ((double)bb[5] - bb[2] + 1);
    ctx->n_cyc_ub = (size_t)std::min((double)n, range_cells);
    if (total <= 32) return acc_build_cycle_t<uint32_t, Items>(ctx, items, n, use_resident, kc, total);
    return acc_build_cycle_t<uint64_t, Items>(ctx, items, n, use_resident, kc, total);
}

// The same with ABSOLUTE 63-bit cell keys: no cell range has to be known (nothing is read back), and the item count may live
// on the device (n = the host's bound).  The radix plan skips the digits that are constant over the batch.
template <typename Items>
int acc_build_cycle_abs(o3r_ctx* ctx, const Items& items, size_t n, bool use_resident, const uint32_t* n_dev) {
    ctx->n_cyc_ub = 0;
    ctx->h_counters[CNT_CYC] = ctx->h_counters[CNT_NEW] = 0;
    if (n == 0) return O3R_OK;
    { int rc = refresh_nres(ctx, false); if (rc) return rc; }
    if (n >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "batch too large for 32-bit indices");
    KeyCodec kc;
    kc.imin = kc.jmin = kc.kmin = -(1 << 20);
    kc.wi = kc.wj = 21;
    ctx->n_cyc_ub = n;
    return acc_build_cycle_t<uint64_t, Items>(ctx, items, n, use_resident, kc, 63, n_dev);
}

// Applies the cycle's cell list to the resident shard: in-place update of found cells, sorted insert of new ones.
// Entirely device-driven: the cycle's cell count, the number of new cells and the resident count are read from device
// memory, launches and buffers are sized by host-known upper bounds, and nothing here waits for the GPU.
int acc_apply_cycle(o3r_ctx* ctx) {
    const size_t n_cyc_ub = ctx->n_cyc_ub;
    if (n_cyc_ub == 0) return O3R_OK;
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    const int cur = ctx->res_cur, nxt = cur ^ 1;
    const uint32_t tiles = cdiv(n_cyc_ub, kTileV);
    const size_t tot_ub = ctx->n_res_ub + n_cyc_ub;
    Tr tr("acc_apply");
    if (tot_ub >= (1ull << 32)) return ctx->fail(O3R_ERR_NOMEM, "resident shard could exceed 2^32 cells");
    CU(ctx->new_cnt.ensure((size_t)tiles * 4));
    CU(ctx->new_off.ensure((size_t)tiles * 4));
    // the shard grows a little every cycle: reserve in big steps (>= 4 M cells, doubling), a reallocation is a
    // cudaMalloc + cudaFree = a device-wide sync of several ms in the middle of the cycle
    if (ctx->res_keys[nxt].cap < tot_ub * 8 || ctx->res_acc[nxt].cap < tot_ub * 16 || ctx->res_rgb[nxt].cap < tot_ub * 16) {
        const size_t cells = std::max<size_t>(2 * tot_ub, (size_t)1 << 22);
        CU(ctx->res_keys[nxt].ensure(cells * 8));
        CU(ctx->res_acc[nxt].ensure(cells * 16));
        CU(ctx->res_rgb[nxt].ensure(cells * 16));
    }
    CU(ctx->new_keys.ensure(n_cyc_ub * 8));
    { int rc = chg_reserve(ctx, n_cyc_ub); if (rc) return rc; }
    if (tr.on) fprintf(stderr, "[o3r trace] n_res_ub %zu n_cyc_ub %zu\n", ctx->n_res_ub, n_cyc_ub);
    tr.mark("ensures");
    LAUNCH(k_acc_update, tiles, kThreads, 0, cnt + CNT_CYC, ctx->cacc.as<float4>(), ctx->crgb.as<uint4>(),
           ctx->res_acc[cur].as<float4>(), ctx->res_rgb[cur].as<uint4>(), ctx->new_cnt.as<uint32_t>());
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->new_cnt.as<uint32_t>(), ctx->new_off.as<uint32_t>(), tiles,
           cnt + CNT_NEWSCAN);
    LAUNCH(k_acc_place_new, tiles, kThreads, 0, cnt + CNT_CYC, ctx->ckey.as<uint64_t>(), ctx->cacc.as<float4>(),
           ctx->crgb.as<uint4>(), ctx->new_off.as<uint32_t>(), ctx->res_keys[cur].as<uint64_t>(), cnt + CNT_NRES,
           ctx->res_keys[nxt].as<uint64_t>(), ctx->res_acc[nxt].as<float4>(), ctx->res_rgb[nxt].as<uint4>(),
           ctx->new_keys.as<uint64_t>());
    if (ctx->n_res_ub) {
        const uint32_t g = std::min<uint32_t>(cdiv(ctx->n_res_ub, kThreads), 148 * 16);
        LAUNCH(k_acc_place_old, g, kThreads, 0, cnt + CNT_NRES, ctx->res_keys[cur].as<uint64_t>(),
               ctx->res_acc[cur].as<float4>(), ctx->res_rgb[cur].as<uint4>(), ctx->new_keys.as<uint64_t>(), cnt + CNT_NEW,
               ctx->res_keys[nxt].as<uint64_t>(), ctx->res_acc[nxt].as<float4>(), ctx->res_rgb[nxt].as<uint4>());
    }
    LAUNCH(k_acc_finish, 1, 32, 0, cnt + CNT_NRES, cnt + CNT_NEW);
    ctx->res_cur = nxt;
    ctx->n_res_ub = tot_ub;
    ctx->n_res_exact = false;
    CU(cudaMemcpyAsync(ctx->h_nres, cnt + CNT_NRES, 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaEventRecord(ctx->ev_nres, ctx->st));
    tr.mark("launches");
    return chg_cycle(ctx, n_cyc_ub);
}

int acc_merge_points(o3r_ctx* ctx, const float4* pts, size_t n, const int* bb) {
    AccItemsPts items{pts, nullptr, nullptr};
    int rc = acc_build_cycle(ctx, items, n, true, bb);
    if (rc) return rc;
    return acc_apply_cycle(ctx);
}

int acc_merge_cells(o3r_ctx* ctx, const o3r_cell* cells, size_t n, const int* bb) {
    AccItemsCells items{cells, nullptr, nullptr};
    int rc = acc_build_cycle(ctx, items, n, true, bb);
    if (rc) return rc;
    return acc_apply_cycle(ctx);
}

int cloud_append_dev(o3r_ctx* ctx, const float4* pts, size_t n) {
    if (n == 0) return O3R_OK;
    CU(ctx->cloud.ensure((ctx->n_cloud + n) * 16, ctx->st, ctx->n_cloud * 16));
    CU(cudaMemcpyAsync(ctx->cloud.as<float4>() + ctx->n_cloud, pts, n * 16, cudaMemcpyDeviceToDevice, ctx->st));
    ctx->n_cloud += n;
    return O3R_OK;
}

}  // namespace
