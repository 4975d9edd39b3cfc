// host_retain.cuh — the sharded RETAIN downsample (the exchange inside the library for O3R_MERGE_RETAIN): every rank keeps the
// points of its own frames, o3r_cloud_transform stays local, and o3r_cloud_downsample is a collective that sends each point once
// to the owner of its combined-grid cell.  The owner sums its cells' points in the single-GPU order, so the union of the shards
// is the single-GPU output bit for bit.  (host side of libo3r.so; included by o3r_api.cu, one translation unit)
//
// Steps of one collective downsample, on every rank:
//   1. local z-shifted bbox -> all-reduce (max) with the frame / cycle ranges and a status word -> global GridParams (sync)
//   2. per point: owner, order tag; one stable radix pass on the owner -> one send buffer of {point, tag} buckets
//   3. counts agreement: grouped send/recv of the per-destination counts + status (sync); receive buffers; all-reduce of
//      "every rank has its buffers" (sync); grouped send/recv of the variable-size buckets
//   4. owner: stable sort of the received records by tag, gather (cloud_big order), k_vg_key + vg_sorted_reduce (engine 1)
// A rank that fails locally still takes part in every agreement step with its error bit set, so all ranks return the error
// and none waits in a receive that is never matched.
#pragma once

#include "host_comm.cuh"
#include "retain.cuh"

namespace {

// (named phases for o3r_profile_read: the split of the collective into local prep, exchange and owner reduction)
cudaEvent_t rt_phase_begin(o3r_ctx* ctx) {
    if (!ctx->profiling) return nullptr;
    cudaEvent_t e = ctx->ev_get();
    cudaEventRecord(e, ctx->st);
    return e;
}
void rt_phase_end(o3r_ctx* ctx, const char* name, cudaEvent_t a) {
    if (!a) return;
    cudaEvent_t b = ctx->ev_get();
    cudaEventRecord(b, ctx->st);
    ctx->prof.push_back({name, a, b});
}

inline uint32_t rt_bits(uint32_t v) { uint32_t b = 0; while (v) { ++b; v >>= 1; } return b; }

// engine 1 over `n` points with the global grid already in ctx->grids (z shifted by 500, the combined grid) -> ctx->rt_out
int rt_engine1(o3r_ctx* ctx, const float4* pts, size_t n, size_t* m) {
    *m = 0;
    if (n == 0) return O3R_OK;
    CU(ctx->rt_out.ensure(n * 16));
    const uint32_t seg_h[2] = {0u, (uint32_t)n};
    { int rcu = upload_small(ctx, ctx->seg2.p, seg_h, 8); if (rcu) return rcu; }
    return vg_one_segment(ctx, pts, ctx->seg2.as<uint32_t>(), n, ctx->inv_c, ctx->inv_c, ctx->inv_cz,
                          ctx->p.min_points_per_voxel, 1, ctx->rt_out.as<float4>(), nullptr, nullptr, m);
}

// step 1, local part: the z-shifted bbox of the local cloud and the words of the first agreement
int rt_local_bbox(o3r_ctx* ctx, uint32_t n_frames, uint32_t* w) {
    const size_t n = ctx->n_cloud;
    if (n > kRtMaxPoints) return ctx->fail(O3R_ERR_INVALID, "local cloud too large for 32-bit indices");
    if (n && ctx->rt_frames.empty()) return ctx->fail(O3R_ERR_INVALID, "retained points without a frame record");
    FILL(ctx->bbox.as<uint32_t>(), 24, FILL_BBOX);
    if (n) {
        const uint32_t seg_h[2] = {0u, (uint32_t)n};
        { int rcu = upload_small(ctx, ctx->seg2.p, seg_h, 8); if (rcu) return rcu; }
        LAUNCH(k_bbox_pts, dim3(cdiv(n, kTileV), 1), kThreads, 0, ctx->cloud.as<float4>(), ctx->seg2.as<uint32_t>(), 1,
               ctx->bbox.as<uint32_t>());
    }
    LAUNCH(k_rt_agree_pack, 1, 32, 0, ctx->bbox.as<uint32_t>(), n_frames, ctx->rt_cycles, 0u, w);
    return O3R_OK;
}

// step 2, local part: owner + tag per point, stable bucketing by owner into ctx->rt_send; counts land in `ocnt`
int rt_route(o3r_ctx* ctx, uint32_t fbits, uint32_t** ocnt_out) {
    const uint32_t world = (uint32_t)ctx->world;
    const size_t n = ctx->n_cloud;
    CU(ctx->okeys.ensure((size_t)kMaxPasses * kRsBins * 4 + sizeof(SortPlan)));
    uint32_t* ocnt = ctx->okeys.as<uint32_t>();
    *ocnt_out = ocnt;
    ZERO(ocnt, (size_t)kMaxPasses * kRsBins * 4);
    if (n == 0) return O3R_OK;
    // the device copy of the frame table grows with the cloud: only the records added since the last downsample are copied
    const size_t nf = ctx->rt_frames.size(), done = std::min(ctx->rt_ftab_n, nf);
    if (nf > done) {
        std::vector<RtFrameDev> tail(nf - done);
        for (size_t i = done; i < nf; ++i) {
            const o3r_ctx::RtFrame& f = ctx->rt_frames[i];
            tail[i - done] = {(uint32_t)f.first, f.cycle, f.frame};
        }
        CU(ctx->rt_ftab.ensure(nf * sizeof(RtFrameDev), ctx->st, done * sizeof(RtFrameDev)));
        CU(cudaMemcpyAsync(ctx->rt_ftab.as<RtFrameDev>() + done, tail.data(), tail.size() * sizeof(RtFrameDev), cudaMemcpyHostToDevice, ctx->st));
        ctx->rt_ftab_n = nf;
    }
    CU(ctx->rt_tags.ensure(n * 4));
    CU(ctx->rt_send.ensure(n * sizeof(RtRec)));
    SortU32 sb;
    int rc = carve_sort_u32(ctx, n, sb);
    if (rc) return rc;
    const uint32_t seg_h[2] = {0u, (uint32_t)n};
    { int rcu = upload_small(ctx, ctx->seg2.p, seg_h, 8); if (rcu) return rcu; }
    SortPlan* plan = reinterpret_cast<SortPlan*>(ocnt + kMaxPasses * kRsBins);
    SortPlan pl;
    memset(&pl, 0, sizeof(pl));
    pl.active_mask = 1; pl.final_parity = 1; pl.n_active = 1; pl.n_passes = 1; pl.bits[0] = 8;
    { int rcu = upload_small(ctx, plan, &pl, sizeof(pl)); if (rcu) return rcu; }
    const uint32_t g = std::min<uint32_t>(cdiv(n, kThreads), 148 * 8);
    LAUNCH(k_rt_route, g, kThreads, 0, ctx->cloud.as<float4>(), (uint32_t)n, ctx->rt_ftab.as<RtFrameDev>(), (uint32_t)nf, fbits,
           ctx->inv_c, ctx->inv_c, ctx->inv_cz, world, sb.k0, ctx->rt_tags.as<uint32_t>(), ocnt);
    rc = sort_pairs<uint32_t>(ctx, sb.k0, sb.k1, sb.v0, sb.v1, ctx->seg2.as<uint32_t>(), 1, n, plan, 1, 1, ocnt, 0);
    if (rc) return rc;
    LAUNCH(k_rt_pack, g, kThreads, 0, ctx->cloud.as<float4>(), ctx->rt_tags.as<uint32_t>(), sb.v1, (uint32_t)n,
           ctx->rt_send.as<RtRec>());
    return O3R_OK;
}

// step 4: the owner's points in cloud_big order, then engine 1 with the global grid
int rt_owner_reduce(o3r_ctx* ctx, size_t n_own, uint32_t tag_bits, size_t* m) {
    *m = 0;
    if (n_own == 0) return O3R_OK;
    const RtRec* rec = ctx->rt_recv.as<RtRec>();
    CU(ctx->rt_pts.ensure(n_own * 16));
    const uint32_t seg_h[2] = {0u, (uint32_t)n_own};
    { int rcu = upload_small(ctx, ctx->seg2.p, seg_h, 8); if (rcu) return rcu; }
    const uint32_t* seg = ctx->seg2.as<uint32_t>();
    SortU32 sb;
    int rc = carve_sort_u32(ctx, n_own, sb);
    if (rc) return rc;
    const uint32_t g = std::min<uint32_t>(cdiv(n_own, kThreads), 148 * 8);
    LAUNCH(k_rt_tags, g, kThreads, 0, rec, (uint32_t)n_own, sb.k0);
    // stable LSD sort on the tag's live bits (passes whose digit is constant are skipped)
    const size_t gh_bytes = (size_t)kMaxPasses * kRsBins * 4;
    CU(ctx->ghist.ensure(gh_bytes));
    CU(ctx->plan_all.ensure(sizeof(SortPlan)));
    ZERO(ctx->ghist.p, gh_bytes);
    SortPlan* plan = ctx->plan_all.as<SortPlan>();
    LAUNCH(k_rs_layout, 1, 64, 0, 1, nullptr, (int)std::max(1u, tag_bits), plan);
    LAUNCH_N("k_rs_ghist_u32", (k_rs_ghist<uint32_t, 4>), dim3(std::max(1u, cdiv(n_own, kRsTile)), 1), kThreads, 0, sb.k0, seg, plan,
             ctx->ghist.as<uint32_t>());
    LAUNCH(k_rs_plan, 1, kThreads, 0, ctx->ghist.as<uint32_t>(), seg, plan, nullptr);
    rc = sort_pairs<uint32_t>(ctx, sb.k0, sb.k1, sb.v0, sb.v1, seg, 1, n_own, plan, 4, 1, ctx->ghist.as<uint32_t>());
    if (rc) return rc;
    LAUNCH(k_rt_gather, g, kThreads, 0, rec, (uint32_t)n_own, plan, sb.v0, sb.v1, ctx->rt_pts.as<float4>());
    return rt_engine1(ctx, ctx->rt_pts.as<float4>(), n_own, m);
}

// every rank leaves the collective with an error: the failing rank with its own, the others naming the peer
int rt_collective_fail(o3r_ctx* ctx, int local_rc, const std::string& local_err) {
    if (local_rc) return ctx->fail(local_rc, "sharded downsample: " + local_err);
    return ctx->fail(O3R_ERR_CUDA, "sharded downsample: a peer rank failed; no rank returns a result");
}

// agreement words written by a copy from the host: the path a rank takes after a local failure (no kernel involved)
int rt_put_words(o3r_ctx* ctx, uint32_t* dst, const uint32_t* src, size_t n_words) {
    CU(cudaMemcpyAsync(dst, src, n_words * 4, cudaMemcpyHostToDevice, ctx->st));
    return O3R_OK;
}

// the first agreement's result on the host: global bbox -> GridParams on the device (k_rt_grid), words + grid read back
int rt_read_verdict(o3r_ctx* ctx, uint32_t* w, uint32_t* hw, GridParams* G) {
    LAUNCH(k_rt_grid, 1, 32, 0, w, ctx->inv_c, ctx->inv_c, ctx->inv_cz, ctx->bbox.as<uint32_t>(), ctx->grids.as<GridParams>());
    CU(cudaMemcpyAsync(hw, w, kRtWords * 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(G, ctx->grids.p, sizeof(GridParams), cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    return O3R_OK;
}

// o3r_cloud_downsample while a communicator is attached to a RETAIN context (not dont_downsample): *res / *m = this rank's
// cells in ascending PCL voxel index (or, on a pass-through grid, its own points).  Collective over the communicator.
//
// Every rank runs the same agreement steps whatever happened locally: a local failure (a limit, an allocation, a launch) only
// sets its status word, and the decision that follows each agreement is taken from the agreed words, so all ranks take it
// alike.  What ends a rank's part early is an NCCL call that fails or a stream that no longer runs (a read-back of an agreement
// fails): the communicator is then unusable for every rank and the caller's recourse is NCCL's own (ncclCommAbort).
int retain_downsample_sharded(o3r_ctx* ctx, const float4** res, size_t* m) {
    *res = ctx->rt_out.as<float4>(); *m = 0;
    if (ctx->rt_valid) { *m = ctx->rt_m; return O3R_OK; }   // the local cloud has not changed since: no communication
    NcclApi* N = nccl_api();
    const uint32_t world = (uint32_t)ctx->world, rank = (uint32_t)ctx->rank;
    ncclComm_t comm = (ncclComm_t)ctx->comm;
    uint32_t* w = ctx->rt_agree.as<uint32_t>();
    uint32_t* csend = w + kRtWords;
    uint32_t* crecv = csend + 2 * world;
    uint32_t* bstat = crecv + 2 * world;
    int local_rc = 0;
    std::string local_err;
    auto local = [&](int rc) { if (rc && !local_rc) { local_rc = rc; local_err = ctx->err; } return rc; };

    // ---- 1. global bbox, frame / cycle ranges and status: one all-reduce (max)
    cudaEvent_t ph = rt_phase_begin(ctx);
    uint32_t n_frames = 0;
    for (const o3r_ctx::RtFrame& f : ctx->rt_frames) n_frames = std::max(n_frames, f.frame + 1);
    if (local(rt_local_bbox(ctx, n_frames, w))) {
        ctx->fq.clear();   // (fills of the failed step: nothing reads them)
        uint32_t e[kRtWords] = {};
        e[RT_W_ERR] = 1;
        { int rcu = rt_put_words(ctx, w, e, kRtWords); if (rcu) return rcu; }
    }
    NC(N->AllReduce(w, w, kRtWords, ncclUint32, ncclMax, comm, ctx->st));
    uint32_t hw[kRtWords] = {};
    GridParams G;
    memset(&G, 0, sizeof(G));
    uint32_t status = local(rt_read_verdict(ctx, w, hw, &G)) ? 1u : 0u;
    // what the agreed words say (identical on every rank that could read them)
    enum { V_EXCHANGE, V_EMPTY, V_PASS, V_FAILED, V_WRAP, V_TAG } verdict = V_EXCHANGE;
    if (status || hw[RT_W_ERR]) verdict = V_FAILED;
    else if (G.empty) verdict = V_EMPTY;
    else if (G.passthrough) verdict = V_PASS;     // PCL returns the input unchanged: every rank keeps its own points
    else if (hw[RT_W_WRAP]) verdict = V_WRAP;
    // order tag = cycle << fbits | global frame index: cloud_big order; its width is agreed, so all ranks check the same limit
    const uint32_t fbits = rt_bits(hw[RT_W_FRAMES] ? hw[RT_W_FRAMES] - 1 : 0), sbits = rt_bits(hw[RT_W_CYCLES] ? hw[RT_W_CYCLES] - 1 : 0);
    if (verdict == V_EXCHANGE && fbits + sbits > 32) verdict = V_TAG;

    // ---- 2. owner + tag per point, stable bucketing by owner
    uint32_t* ocnt = ctx->okeys.as<uint32_t>();
    if (verdict == V_EXCHANGE && local(rt_route(ctx, fbits, &ocnt))) status = 1;
    rt_phase_end(ctx, "retain_prep", ph);

    // ---- 3. counts agreement (every verdict: a rank that could not read the first one says so here), buffer agreement,
    //      exchange of the buckets
    ph = rt_phase_begin(ctx);
    bool counts_written = false;
    if (verdict == V_EXCHANGE && !status) {
        if (fill_flush(ctx) == O3R_OK) {
            k_rt_counts<<<1, kThreads, 0, ctx->st>>>(ocnt, world, csend);   // (not LAUNCH: a failure must not return)
            ++ctx->launches;
            counts_written = cudaGetLastError() == cudaSuccess;
        }
        if (!counts_written) { status = 1; local(ctx->fail(O3R_ERR_CUDA, "k_rt_counts launch failed")); }
    }
    if (!counts_written) {
        ctx->fq.clear();
        std::vector<uint32_t> zc(2 * (size_t)world, 0u);
        for (uint32_t d = 0; d < world; ++d) zc[2 * d + 1] = status;
        { int rcu = rt_put_words(ctx, csend, zc.data(), zc.size()); if (rcu) return rcu; }
    }
    CU(cudaMemcpyAsync(crecv + 2 * rank, csend + 2 * rank, 8, cudaMemcpyDeviceToDevice, ctx->st));
    if (world > 1) {
        ncclResult_t r = N->GroupStart();
        if (r != ncclSuccess) return ctx->fail(O3R_ERR_CUDA, std::string("NCCL error at GroupStart: ") + N->GetErrorString(r));
        for (uint32_t peer = 0; peer < world && r == ncclSuccess; ++peer) {
            if (peer == rank) continue;
            r = N->Send(csend + 2 * peer, 2, ncclUint32, (int)peer, comm, ctx->st);
            if (r == ncclSuccess) r = N->Recv(crecv + 2 * peer, 2, ncclUint32, (int)peer, comm, ctx->st);
        }
        const ncclResult_t re = N->GroupEnd();
        if (r == ncclSuccess) r = re;
        if (r != ncclSuccess) return ctx->fail(O3R_ERR_CUDA, std::string("NCCL error in the counts agreement: ") + N->GetErrorString(r));
    }
    std::vector<uint32_t> hc(4 * (size_t)world);   // [world][2] sent, [world][2] received
    CU(cudaMemcpyAsync(hc.data(), csend, hc.size() * 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    std::vector<size_t> scnt(world), rcnt(world), soff(world + 1, 0), roff(world + 1, 0);
    bool peer_failed = false;
    for (uint32_t d = 0; d < world; ++d) {
        scnt[d] = hc[2 * d];
        rcnt[d] = hc[2 * world + 2 * d];
        peer_failed = peer_failed || hc[2 * world + 2 * d + 1];
        soff[d + 1] = soff[d] + scnt[d];
        roff[d + 1] = roff[d] + rcnt[d];
    }
    if (peer_failed || verdict == V_FAILED) return rt_collective_fail(ctx, local_rc, local_err);
    if (verdict == V_WRAP) return ctx->fail(O3R_ERR_UNSUPPORTED, "sharded downsample: the combined grid has more than 2^32 cells");
    if (verdict == V_TAG)
        return ctx->fail(O3R_ERR_UNSUPPORTED, "sharded downsample: cycles x frames per cycle exceed the 32-bit order tag; clear the cloud");
    if (verdict == V_EMPTY) { ctx->rt_valid = true; ctx->rt_m = 0; rt_phase_end(ctx, "retain_exchange", ph); return O3R_OK; }
    if (verdict == V_PASS) {   // no further communication
        int rc = rt_engine1(ctx, ctx->cloud.as<float4>(), ctx->n_cloud, m);
        if (rc) return rc;
        ctx->rt_valid = true; ctx->rt_m = *m;
        *res = ctx->rt_out.as<float4>();
        rt_phase_end(ctx, "retain_exchange", ph);
        return O3R_OK;
    }
    const size_t n_own = roff[world];
    // receive buffers; then "every rank has its buffers"
    uint32_t bufs_bad = 0;
    if (n_own > kRtMaxPoints) { bufs_bad = 1; local(ctx->fail(O3R_ERR_INVALID, "owned points exceed the 32-bit index range")); }
    else {
        cudaError_t e = ctx->rt_recv.ensure(std::max<size_t>(n_own, 1) * sizeof(RtRec));
        if (e != cudaSuccess) { bufs_bad = 1; local(ctx->fail_cuda(e, "rt_recv.ensure", __FILE__, __LINE__)); }
    }
    { int rcu = rt_put_words(ctx, bstat, &bufs_bad, 1); if (rcu) return rcu; }
    NC(N->AllReduce(bstat, bstat, 1, ncclUint32, ncclMax, comm, ctx->st));
    uint32_t any_bad = 0;
    CU(cudaMemcpyAsync(&any_bad, bstat, 4, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    if (any_bad) return rt_collective_fail(ctx, local_rc, local_err);
    const char* snd = ctx->rt_send.as<char>();
    char* rcv = ctx->rt_recv.as<char>();
    constexpr size_t R = sizeof(RtRec);
    if (scnt[rank]) CU(cudaMemcpyAsync(rcv + roff[rank] * R, snd + soff[rank] * R, scnt[rank] * R, cudaMemcpyDeviceToDevice, ctx->st));
    if (world > 1) {   // both sides of a pair know its size: empty buckets are skipped on both
        ncclResult_t r = N->GroupStart();
        if (r != ncclSuccess) return ctx->fail(O3R_ERR_CUDA, std::string("NCCL error at GroupStart: ") + N->GetErrorString(r));
        for (uint32_t peer = 0; peer < world && r == ncclSuccess; ++peer) {
            if (peer == rank) continue;
            if (scnt[peer]) r = N->Send(snd + soff[peer] * R, scnt[peer] * R, ncclChar, (int)peer, comm, ctx->st);
            if (r == ncclSuccess && rcnt[peer]) r = N->Recv(rcv + roff[peer] * R, rcnt[peer] * R, ncclChar, (int)peer, comm, ctx->st);
        }
        const ncclResult_t re = N->GroupEnd();
        if (r == ncclSuccess) r = re;
        if (r != ncclSuccess) return ctx->fail(O3R_ERR_CUDA, std::string("NCCL error in the point exchange: ") + N->GetErrorString(r));
    }
    rt_phase_end(ctx, "retain_exchange", ph);

    // ---- 4. owner reduction (no further communication)
    ph = rt_phase_begin(ctx);
    int rc = rt_owner_reduce(ctx, n_own, fbits + sbits, m);
    if (rc) return rc;
    rt_phase_end(ctx, "retain_reduce", ph);
    ctx->rt_valid = true; ctx->rt_m = *m;
    *res = ctx->rt_out.as<float4>();
    return O3R_OK;
}

}  // namespace
