// host_comm.cuh — the multi-GPU exchange inside the library (SURVEY 8e): one process per GPU, a cycle's partial cells are
// hash-partitioned by owner rank and exchanged with grouped ncclSend / ncclRecv (= all-to-all) on the context's stream,
// then folded into the rank's shard.  Nothing in a cycle's exchange waits for the GPU: every (source, destination) pair
// moves one fixed-size slot whose first record carries the number of valid cells, so no split sizes cross the host.
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
//
// NCCL is bound at run time (dlopen of libnccl.so.2): libo3r.so has no link-time dependency on it, a process that already
// loaded NCCL (PyTorch) shares that copy, and single-GPU users never touch it.
#pragma once

#include <dlfcn.h>
#include <nccl.h>

#include "host_merge.cuh"

namespace o3r {

// the pre-reduced cycle list (ckey / cacc / crgb, in owner order through `order`; the cell count lives on the device) ->
// fixed-size slots: slot d = [header | slot_cap cells]; header.key = valid cells.  counts[d] = cells owned by d (raw
// histogram); a slot that would overflow raises *xflag and is truncated.
__global__ void __launch_bounds__(kThreads) k_pack_slots_cyc(const uint32_t* __restrict__ n_cyc_ptr, const uint32_t* __restrict__ order,
                                                             const uint64_t* __restrict__ ckey, const float4* __restrict__ cacc,
                                                             const uint4* __restrict__ crgb, const uint32_t* __restrict__ counts,
                                                             uint32_t world, uint32_t slot_cap, o3r_cell* __restrict__ slots,
                                                             uint32_t* __restrict__ xflag) {
    __shared__ uint32_t s_start[257];
    const uint32_t n = *n_cyc_ptr;
    if (threadIdx.x == 0) {
        uint32_t a = 0;
        for (uint32_t d = 0; d < world; ++d) { s_start[d] = a; a += counts[d]; }
        s_start[world] = a;
    }
    __syncthreads();
    if (blockIdx.x == 0)
        for (uint32_t d = threadIdx.x; d < world; d += kThreads) {
            o3r_cell h;
            h.key = min(counts[d], slot_cap); h.sx = h.sy = h.sz = 0.f; h.n = h.sr = h.sg = h.sb = h.pad = 0u;
            slots[(size_t)d * (slot_cap + 1)] = h;
            if (counts[d] > slot_cap) atomicOr(xflag, 1u);
        }
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        uint32_t d = 0;   // owner of position i of the owner-sorted list
        while (d + 1 < world && s_start[d + 1] <= i) ++d;
        const uint32_t at = i - s_start[d];
        if (at < slot_cap) {
            const uint32_t h = order[i];
            const float4 a = cacc[h];
            const uint4 c = crgb[h];
            o3r_cell r;
            r.key = ckey[h];
            r.sx = a.x; r.sy = a.y; r.sz = a.z; r.n = __float_as_uint(a.w);
            r.sr = c.x; r.sg = c.y; r.sb = c.z; r.pad = 0u;
            slots[(size_t)d * (slot_cap + 1) + 1 + at] = r;
        }
    }
}

// received slots (one per source rank, in rank order) -> contiguous list + count, all on the device
__global__ void __launch_bounds__(kThreads) k_unpack_slots(const o3r_cell* __restrict__ slots, uint32_t world, uint32_t slot_cap,
                                                           o3r_cell* __restrict__ out, uint32_t* __restrict__ n_out) {
    __shared__ uint32_t s_start[257];
    if (threadIdx.x == 0) {
        uint32_t a = 0;
        for (uint32_t s = 0; s < world; ++s) { s_start[s] = a; const unsigned long long c = slots[(size_t)s * (slot_cap + 1)].key; a += c < slot_cap ? (uint32_t)c : slot_cap; }
        s_start[world] = a;
        if (blockIdx.x == 0) *n_out = a;
    }
    __syncthreads();
    const uint32_t n = s_start[world];
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        uint32_t s = 0;
        while (s + 1 < world && s_start[s + 1] <= i) ++s;
        out[i] = slots[(size_t)s * (slot_cap + 1) + 1 + (i - s_start[s])];
    }
}

}  // namespace o3r

namespace {

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string err;
};

NcclApi* nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (!api.lib) { api.err = std::string("cannot load libnccl.so.2: ") + dlerror(); return; }
        auto sym = [&](const char* n) { void* p = dlsym(api.lib, n); if (!p && api.err.empty()) api.err = std::string("libnccl lacks ") + n; return p; };
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
        api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
        api.Send = reinterpret_cast<decltype(api.Send)>(sym("ncclSend"));
        api.Recv = reinterpret_cast<decltype(api.Recv)>(sym("ncclRecv"));
        api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    });
    return &api;
}

#define NC(call)                                                                                      \
    do {                                                                                              \
        if (ctx->fq.L.n) { int rcf_ = fill_flush(ctx); if (rcf_) return rcf_; }                       \
        ncclResult_t r_ = (call);                                                                     \
        if (r_ != ncclSuccess)                                                                        \
            return ctx->fail(O3R_ERR_CUDA, std::string("NCCL error at " #call ": ") + N->GetErrorString(r_)); \
    } while (0)

int comm_setup(o3r_ctx* ctx, int world, int rank, size_t slot_cells) {
    if (world < 1 || world > 256 || rank < 0 || rank >= world || slot_cells == 0 || slot_cells >= (1ull << 31))
        return ctx->fail(O3R_ERR_INVALID, "bad communicator arguments");
    if (ctx->retain()) {   // RETAIN / dont_downsample: the points stay where they are made (host_retain.cuh); no slots
        if (ctx->n_cloud) return ctx->fail(O3R_ERR_INVALID, "a sharded retained cloud starts empty: attach the communicator before the first cycle");
        CU(ctx->rt_agree.ensure(((size_t)16 + 4 * (size_t)world + 4) * 4));
        CU(ctx->seg2.ensure(16));   // (these four are what the downsample's agreement steps touch: they never fail later)
        CU(ctx->bbox.ensure(6 * 4));
        CU(ctx->grids.ensure(sizeof(GridParams)));
        ctx->world = world; ctx->rank = rank; ctx->slot_cap = (uint32_t)slot_cells;
        ctx->rt_reset();
        return O3R_OK;
    }
    ctx->world = world; ctx->rank = rank; ctx->slot_cap = (uint32_t)slot_cells;
    const size_t bytes = (size_t)world * (slot_cells + 1) * sizeof(o3r_cell);
    CU(ctx->x_send.ensure(bytes));
    CU(ctx->x_recv.ensure(bytes));
    CU(ctx->x_list.ensure((size_t)world * slot_cells * sizeof(o3r_cell)));
    return O3R_OK;
}

// One cycle's exchange, queued on the context's stream: bucket the last batch's partial cells by owner, all-to-all of the
// fixed-size slots, merge what arrived.  Collective over the communicator; returns without waiting for the GPU.
int exchange_cycle_impl(o3r_ctx* ctx) {
    NcclApi* N = nccl_api();
    if (!ctx->comm) return ctx->fail(O3R_ERR_INVALID, "no communicator: call o3r_comm_init / o3r_comm_attach first");
    const uint32_t world = (uint32_t)ctx->world, cap = ctx->slot_cap;
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    // ---- this rank's cycle, pre-reduced on the combined grid (sort by compact cell key + in-order partial sums against an empty
    //      resident: voxel.cuh engine 2): the cycle's frames overlap, so ~8x fewer records cross NVLink and reach the owners' merge
    size_t nub = 0;
    if (ctx->last_is_vox && ctx->last_total) {
        const int* bbp = ctx->last_has_cellbb ? ctx->last_cellbb : nullptr;
        int rc;
        if (ctx->last_has_partials) {
            AccItemsCells items{ctx->partials.as<o3r_cell>(), nullptr, nullptr};
            rc = acc_build_cycle(ctx, items, ctx->last_partials, false, bbp);
        } else {   // exact-order modes keep the batch as voxel points
            AccItemsPts items{ctx->vox.as<float4>(), nullptr, nullptr};
            rc = acc_build_cycle(ctx, items, ctx->last_total, false, bbp);
        }
        if (rc) return rc;
        nub = ctx->n_cyc_ub;
    } else {
        ZERO(cnt + CNT_CYC, 4);
    }
    // ---- bucket by owner: one stable radix pass on the owner id (a rank's cells stay in key order inside a slot)
    CU(ctx->okeys.ensure((size_t)kMaxPasses * kRsBins * 4 + sizeof(SortPlan)));
    uint32_t* ocnt = ctx->okeys.as<uint32_t>();
    ZERO(ocnt, (size_t)kMaxPasses * kRsBins * 4);
    SortU32 sb{nullptr, nullptr, nullptr, nullptr};
    CU(ctx->seg2.ensure(16));
    const uint32_t g = std::min<uint32_t>(std::max(1u, cdiv(nub, kThreads)), 148 * 8);
    if (nub) {
        int rc = carve_sort_u32(ctx, nub, sb);
        if (rc) return rc;
        SortPlan* plan = reinterpret_cast<SortPlan*>(ocnt + kMaxPasses * kRsBins);
        SortPlan pl;
        memset(&pl, 0, sizeof(pl));
        pl.active_mask = 1; pl.final_parity = 1; pl.n_active = 1; pl.n_passes = 1; pl.bits[0] = 8;
        { int rcu = upload_small(ctx, plan, &pl, sizeof(pl)); if (rcu) return rcu; }
        LAUNCH(k_owner, g, kThreads, 0, cnt + CNT_CYC, ctx->ckey.as<uint64_t>(), world, sb.k0, sb.v0, ocnt, ctx->seg2.as<uint32_t>());
        rc = sort_pairs<uint32_t>(ctx, sb.k0, sb.k1, sb.v0, sb.v1, ctx->seg2.as<uint32_t>(), 1, nub, plan, 1, 0, ocnt, 0);
        if (rc) return rc;
    }
    LAUNCH(k_pack_slots_cyc, g, kThreads, 0, cnt + CNT_CYC, sb.v1, ctx->ckey.as<uint64_t>(), ctx->cacc.as<float4>(), ctx->crgb.as<uint4>(),
           ocnt, world, cap, ctx->x_send.as<o3r_cell>(), cnt + CNT_XFLAG);
    // ---- all-to-all of the slots
    const size_t slot_bytes = (size_t)(cap + 1) * sizeof(o3r_cell);
    char* snd = ctx->x_send.as<char>();
    char* rcv = ctx->x_recv.as<char>();
    CU(cudaMemcpyAsync(rcv + (size_t)ctx->rank * slot_bytes, snd + (size_t)ctx->rank * slot_bytes, slot_bytes, cudaMemcpyDeviceToDevice, ctx->st));
    if (world > 1) {
        NC(N->GroupStart());
        for (uint32_t peer = 0; peer < world; ++peer) {
            if ((int)peer == ctx->rank) continue;
            NC(N->Send(snd + (size_t)peer * slot_bytes, slot_bytes, ncclChar, (int)peer, (ncclComm_t)ctx->comm, ctx->st));
            NC(N->Recv(rcv + (size_t)peer * slot_bytes, slot_bytes, ncclChar, (int)peer, (ncclComm_t)ctx->comm, ctx->st));
        }
        NC(N->GroupEnd());
    }
    // ---- merge what this rank owns (item count stays on the device; absolute keys: no cell range has to be agreed on)
    const size_t n_ub = (size_t)world * cap;
    LAUNCH(k_unpack_slots, std::min<uint32_t>(cdiv(n_ub, kThreads), 148 * 8), kThreads, 0, ctx->x_recv.as<o3r_cell>(), world, cap,
           ctx->x_list.as<o3r_cell>(), cnt + CNT_XRECV);
    AccItemsCells items{ctx->x_list.as<o3r_cell>(), nullptr, nullptr};
    int rc = acc_build_cycle_abs(ctx, items, n_ub, true, cnt + CNT_XRECV);
    if (rc) return rc;
    rc = acc_apply_cycle(ctx);
    if (rc) return rc;
    ctx->x_pending_check = true;   // the overflow flag is read with the next o3r_cloud_downsample, which waits for the GPU anyway
    return O3R_OK;
}

}  // namespace
