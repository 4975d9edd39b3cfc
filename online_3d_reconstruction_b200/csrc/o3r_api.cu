// o3r_api.cu — C ABI (include/o3r.h) over the sm_100a kernels.  No CPU fallback: every compute entry
// point launches CUDA kernels on the context's stream and fails with O3R_ERR_CUDA otherwise.
#include "host_ctx.cuh"
#include "host_sort.cuh"
#include "host_merge.cuh"
#include "host_sor.cuh"
#include "host_frames.cuh"
#include "host_comm.cuh"
#include "host_retain.cuh"
#include "host_changes.cuh"
#include "host_checkpoint.cuh"
#include "host_register.cuh"
#include "host_mesh.cuh"


// =====================================================================================================================
extern "C" {

int o3r_version(void) { return O3R_VERSION; }

const char* o3r_last_error(const o3r_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int o3r_create(const o3r_params* params, o3r_ctx** out_ctx) {
    if (!params || !out_ctx) { g_create_err = "null argument"; return O3R_ERR_INVALID; }
    *out_ctx = nullptr;
    const o3r_params& p = *params;
    if (p.rows <= 0 || p.cols <= 0 || p.bounding_box < 0 || p.cols_start_aft_cutout < 0 || p.jump_pixels < 0 ||
        !(p.voxel_size > 0) || p.max_batch_frames < 1) {
        g_create_err = "invalid o3r_params";
        return O3R_ERR_INVALID;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= p.device) {
        g_create_err = std::string("no usable CUDA device: ") + cudaGetErrorString(e) + " (there is no CPU fallback)";
        return O3R_ERR_CUDA;
    }
    e = cudaSetDevice(p.device);
    if (e != cudaSuccess) { g_create_err = cudaGetErrorString(e); return O3R_ERR_CUDA; }
    o3r_ctx* ctx = new o3r_ctx();
    ctx->p = p;
    const int J = p.jump_pixels;
    if (J > 0) {  // pose_functions.cpp:1094-1128
        ctx->ny = std::max(0, (p.rows - 2 * p.bounding_box + J - 1) / J);
        ctx->nx = std::max(0, (p.cols - p.bounding_box - p.cols_start_aft_cutout + J - 1) / J);
    }
    ctx->npix = (uint32_t)ctx->nx * (uint32_t)ctx->ny;
    const double* Q = p.Q;
    ctx->canon = Q[1] == 0 && Q[2] == 0 && Q[4] == 0 && Q[6] == 0 && Q[8] == 0 && Q[9] == 0 && Q[10] == 0 &&
                 Q[12] == 0 && Q[13] == 0;
    ctx->leaf_f = (float)(p.voxel_size / 5);          // pose_functions.cpp:1698
    ctx->inv_f = 1.0f / ctx->leaf_f;                  // PCL: inverse_leaf_size_ = Ones / leaf_size_
    ctx->leaf_c = (float)p.voxel_size;                // pose_functions.cpp:1694
    ctx->inv_c = 1.0f / ctx->leaf_c;
    ctx->inv_cz = 1.0f / 1000.0f;
    auto bail = [&](cudaError_t er, const char* what) {
        g_create_err = std::string(what) + ": " + cudaGetErrorString(er);
        o3r_destroy(ctx);
        return O3R_ERR_CUDA;
    };
    if ((e = cudaStreamCreateWithFlags(&ctx->st, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "stream");
    if ((e = cudaStreamCreateWithFlags(&ctx->st_copy, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "stream");
    if ((e = cudaStreamCreateWithFlags(&ctx->st_copy2, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "stream");
    if ((e = cudaEventCreateWithFlags(&ctx->ev_copy2, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "event");
    if (const char* cf = getenv("O3R_CHUNK_FRAMES")) ctx->in.chunk_frames = std::max(1, atoi(cf));
    if (const char* cf = getenv("O3R_CHUNK_FRAMES_DEV")) ctx->in.chunk_frames_dev = std::max(1, atoi(cf));
    if ((e = cudaMallocHost((void**)&ctx->h_counters, CNT_N * 4)) != cudaSuccess) return bail(e, "pinned");
    if ((e = cudaMallocHost((void**)&ctx->res.h_n, 4)) != cudaSuccess) return bail(e, "pinned");
    if ((e = cudaEventCreateWithFlags(&ctx->res.ev_n, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "event");
    if ((e = ctx->counters.ensure(CNT_N * 4)) != cudaSuccess) return bail(e, "counters");
    if ((e = cudaMemsetAsync(ctx->counters.p, 0, CNT_N * 4, ctx->st)) != cudaSuccess) return bail(e, "memset");
    // 1/(q14*d+q15) and (float)(q11 * that) for u8 disparities
    double lr[256];
    float lz[256];
    for (int d = 0; d < 256; ++d) {
        const double v3 = Q[14] * (double)d + Q[15];
        lr[d] = 1.0 / v3;
        lz[d] = (float)(Q[11] * lr[d]);
    }
    if ((e = ctx->lut_r.ensure(sizeof(lr))) != cudaSuccess) return bail(e, "lut");
    if ((e = ctx->lut_z.ensure(sizeof(lz))) != cudaSuccess) return bail(e, "lut");
    cudaMemcpyAsync(ctx->lut_r.p, lr, sizeof(lr), cudaMemcpyHostToDevice, ctx->st);
    cudaMemcpyAsync(ctx->lut_z.p, lz, sizeof(lz), cudaMemcpyHostToDevice, ctx->st);
    if ((e = cudaStreamSynchronize(ctx->st)) != cudaSuccess) return bail(e, "init sync");
    // the radix pass: both key widths, each with the 32-bit and the wide (64-bit) look-back word
    e = cudaFuncSetAttribute(k_rs_onesweep<uint64_t, uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)rs_scatter_smem<uint64_t>());
    if (e != cudaSuccess) return bail(e, "smem attr (is this an sm_100a device?)");
    e = cudaFuncSetAttribute(k_rs_onesweep<uint32_t, uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)rs_scatter_smem<uint32_t>());
    if (e != cudaSuccess) return bail(e, "smem attr");
    e = cudaFuncSetAttribute(k_rs_onesweep<uint64_t, uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)rs_scatter_smem<uint64_t>());
    if (e != cudaSuccess) return bail(e, "smem attr");
    e = cudaFuncSetAttribute(k_rs_onesweep<uint32_t, uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)rs_scatter_smem<uint32_t>());
    if (e != cudaSuccess) return bail(e, "smem attr");
    // shared-memory carve-out per kernel (percent of the 228 KB array; the rest is L1).  Measured on B200:
    // the run-reduce kernels gather points, so they want L1 as much as occupancy.
    cudaFuncSetAttribute(k_vg_reduce_w<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
    cudaFuncSetAttribute(k_vg_reduce_w<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
    cudaFuncSetAttribute(k_acc_reduce<uint32_t, AccItemsPts>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
    cudaFuncSetAttribute(k_acc_reduce<uint64_t, AccItemsPts>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
    cudaFuncSetAttribute(k_acc_reduce<uint32_t, AccItemsCells>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
    cudaFuncSetAttribute(k_acc_reduce<uint64_t, AccItemsCells>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
    cudaFuncSetAttribute(k_rs_onesweep<uint32_t, uint32_t>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_rs_onesweep<uint64_t, uint32_t>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_rs_onesweep<uint32_t, uint64_t>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_rs_onesweep<uint64_t, uint64_t>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    e = cudaFuncSetAttribute(k_bk_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bk_reduce_smem());
    if (e != cudaSuccess) return bail(e, "smem attr");
    // the bucket kernels stage through shared memory and want their 4-5 CTAs per SM: largest carve-out
    cudaFuncSetAttribute(k_bk_reduce, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_bk_scatter<O3R_DISP_U8>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_bk_scatter<O3R_DISP_U16>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_bk_scatter<O3R_DISP_F32>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_bk_scatter<O3R_DISP_F64>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_blur<O3R_BLUR_MEDIAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)blur_smem(kBlurMaxK, O3R_BLUR_MEDIAN));
    cudaFuncSetAttribute(k_blur<O3R_BLUR_BOX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)blur_smem(kBlurMaxK, O3R_BLUR_BOX));
    *out_ctx = ctx;
    return O3R_OK;
}

void o3r_destroy(o3r_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->p.device);
    if (ctx->st_copy2) cudaStreamSynchronize(ctx->st_copy2);
    if (ctx->st_copy) cudaStreamSynchronize(ctx->st_copy);
    if (ctx->st) cudaStreamSynchronize(ctx->st);
    if (ctx->comm && ctx->comm_owned && nccl_api()->CommDestroy) nccl_api()->CommDestroy((ncclComm_t)ctx->comm);
    delete ctx;   // (~o3r_ctx: events, pinned memory, streams, then every device buffer)
}

uint64_t o3r_launch_count(const o3r_ctx* ctx) { return ctx ? ctx->launches : 0; }
size_t o3r_last_batch_partials(const o3r_ctx* ctx) { return (ctx && ctx->last.has_partials) ? ctx->last.n_part : 0; }
int o3r_last_batch_engine(const o3r_ctx* ctx) { return ctx ? (int)ctx->last.engine : 0; }
void* o3r_stream(o3r_ctx* ctx) { return ctx ? (void*)ctx->st : nullptr; }

int o3r_sync(o3r_ctx* ctx) {
    return api(ctx, [&] {
        CU(cudaStreamSynchronize(ctx->st));
        return O3R_OK;
    });
}

int o3r_profile(o3r_ctx* ctx, int enable) {
    return api(ctx, [&] {
        CU(cudaStreamSynchronize(ctx->st));
        for (auto& r : ctx->prof.recs) { ctx->prof.pool.push_back(r.a); ctx->prof.pool.push_back(r.b); }
        ctx->prof.recs.clear();
        ctx->prof.on = enable != 0;
        return O3R_OK;
    });
}

int o3r_profile_read(o3r_ctx* ctx, char* buf, size_t cap) {
    if (!buf || cap == 0) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        CU(cudaStreamSynchronize(ctx->st));
        struct Agg { std::string name; uint64_t n; double ms; };
        std::vector<Agg> agg;
        for (auto& r : ctx->prof.recs) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, r.a, r.b);
            std::string nm = r.name;
            size_t i = 0;
            for (; i < agg.size(); ++i) if (agg[i].name == nm) break;
            if (i == agg.size()) agg.push_back({nm, 0, 0.0});
            agg[i].n += 1; agg[i].ms += ms;
        }
        std::string out;
        char line[256];
        for (auto& a : agg) {
            snprintf(line, sizeof(line), "%s\t%llu\t%.6f\n", a.name.c_str(), (unsigned long long)a.n, a.ms);
            out += line;
        }
        if (out.size() + 1 > cap) return ctx->fail(O3R_ERR_CAPACITY, "profile buffer too small");
        memcpy(buf, out.c_str(), out.size() + 1);
        return O3R_OK;
    });
}

int o3r_set_keep_frame_voxels(o3r_ctx* ctx, int keep) {
    return api(ctx, [&] {
        ctx->keep_frame_voxels = keep != 0;
        return O3R_OK;
    });
}

void* o3r_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
    return p;
}
void o3r_host_free(void* p) { if (p) cudaFreeHost(p); }

int o3r_frames_cloud_dev(o3r_ctx* ctx, const o3r_frame* frames, int n, int disp_type, uint32_t* frame_counts) {
    if (n > 0 && !frames) return O3R_ERR_INVALID;
    return api(ctx, [&] { return frames_cloud_impl(ctx, frames, n, disp_type, frame_counts, BatchOpts(), false); });
}

int o3r_frames_cloud(o3r_ctx* ctx, const o3r_frame* frames, int n, int disp_type, uint32_t* frame_counts) {
    if (n > 0 && !frames) return O3R_ERR_INVALID;
    return api(ctx, [&] { return frames_cloud_impl(ctx, frames, n, disp_type, frame_counts, BatchOpts(), true); });
}

int o3r_frames_prefetch(o3r_ctx* ctx, const o3r_frame* frames, int n, int disp_type) {
    if (n <= 0 || !frames) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (disp_type < 0 || disp_type > 3) return ctx->fail(O3R_ERR_INVALID, "bad disp_type");
        const o3r_params& p = ctx->p;
        const bool label_mode = p.use_segment_labels && frames[0].labels && frames[0].plane_coef;
        for (int i = 0; i < n; ++i)
            if (!frames[i].bgr || (!frames[i].disp && !label_mode) || (label_mode && (!frames[i].labels || !frames[i].plane_coef)))
                return ctx->fail(O3R_ERR_INVALID, "frame without disparity/colour");
        int rc = flush_deferred_prefetch(ctx);   // at most one request waits; an older one goes out now
        if (rc) return rc;
        ctx->in.deferred.frames.assign(frames, frames + n);
        ctx->in.deferred.disp_type = disp_type;
        ctx->in.deferred.pending = true;
        return O3R_OK;
    });
}

int o3r_frames_prefetch_cancel(o3r_ctx* ctx) {
    return api(ctx, [&] {
        ctx->in.deferred.pending = false;           // recorded but not issued: nothing will ever read those buffers
        ctx->in.deferred.frames.clear();
        CU(cudaStreamSynchronize(ctx->st_copy2));   // copies already in flight finish reading the host buffers here
        CU(cudaStreamSynchronize(ctx->st_copy));
        for (auto& pf : ctx->in.prefetch) pf.valid = false;
        return O3R_OK;
    });
}

int o3r_frame_cloud(o3r_ctx* ctx, const o3r_frame* frame, int disp_type, o3r_point* out, size_t cap, size_t* n_out) {
    if (!frame) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (n_out) *n_out = 0;
        BatchOpts opt;
        opt.merge = false;
        int rc = frames_cloud_impl(ctx, frame, 1, disp_type, nullptr, opt, true);
        if (rc) return rc;
        const float4* src = ctx->last.is_vox ? ctx->last.vox.as<float4>() : ctx->last.pts.as<float4>();
        return copy_out(ctx, src, ctx->last.total, out, cap, n_out);
    });
}

int o3r_frame_mask(o3r_ctx* ctx, const o3r_frame* frame, int disp_type, uint8_t* mask, size_t cap, size_t* n_scanned) {
    if (!frame) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (n_scanned) *n_scanned = ctx->npix;
        if (!mask && cap == 0) return O3R_OK;
        if (cap < ctx->npix) return ctx->fail(O3R_ERR_CAPACITY, "mask buffer too small");
        if (ctx->npix == 0) return O3R_OK;
        CU(ctx->mask.ensure(ctx->npix));
        BatchOpts opt;
        opt.merge = false; opt.mask_only = true; opt.mask_dev = ctx->mask.as<uint8_t>();
        int rc = frames_cloud_impl(ctx, frame, 1, disp_type, nullptr, opt, true);
        if (rc) return rc;
        CU(cudaMemcpyAsync(mask, ctx->mask.p, ctx->npix, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
        return O3R_OK;
    });
}

int o3r_last_batch_points(o3r_ctx* ctx, o3r_point* out, size_t cap, size_t* n_out) {
    return api(ctx, [&] {
        if (ctx->last.engine != Engine::SORT && !ctx->keep_frame_voxels)
            return ctx->fail(O3R_ERR_UNSUPPORTED, "O3R_MERGE_ACCUMULATE_FUSED does not materialise the per-frame clouds (see o3r_set_keep_frame_voxels)");
        const float4* src = ctx->last.is_vox ? ctx->last.vox.as<float4>() : ctx->last.pts.as<float4>();
        return copy_out(ctx, src, ctx->last.total, out, cap, n_out);
    });
}

int o3r_cloud_transform(o3r_ctx* ctx, const float T[16]) {
    if (!T) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (!ctx->retain())
            return ctx->fail(O3R_ERR_UNSUPPORTED,
                             "o3r_cloud_transform needs O3R_MERGE_RETAIN: accumulated cells cannot be re-binned");
        ctx->rt.valid = false;   // (on every rank of a sharded cloud, even one without points: the ranks stay in step)
        if (ctx->res.n_cloud == 0) return O3R_OK;
        CU(ctx->tmat.ensure(64));
        { int rcu = upload_small(ctx, ctx->tmat.p, T, 48); if (rcu) return rcu; }
        const uint32_t g = std::min<uint32_t>(cdiv(ctx->res.n_cloud, kThreads), 148 * 16);
        LAUNCH(k_transform_pts, g, kThreads, 0, ctx->res.cloud.as<float4>(), ctx->res.n_cloud, ctx->tmat.as<float>());
        return O3R_OK;
    });
}

int o3r_cloud_append(o3r_ctx* ctx, const o3r_point* pts, size_t n) {
    if (n && !pts) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (ctx->comm && ctx->retain())
            return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_append on a sharded retained cloud: appended points have no place in the frame order");
        if (n == 0) return O3R_OK;
        if (ctx->retain()) {
            CU(ctx->res.cloud.ensure((ctx->res.n_cloud + n) * 16, ctx->st, ctx->res.n_cloud * 16));
            CU(cudaMemcpyAsync(ctx->res.cloud.as<float4>() + ctx->res.n_cloud, pts, n * 16, cudaMemcpyHostToDevice, ctx->st));
            CU(cudaStreamSynchronize(ctx->st));   // the caller may reuse or free `pts` as soon as this returns
            ctx->res.n_cloud += n;
            return O3R_OK;
        }
        CU(ctx->in_pts.ensure(n * 16));
        CU(cudaMemcpyAsync(ctx->in_pts.p, pts, n * 16, cudaMemcpyHostToDevice, ctx->st));
        const int rc = acc_merge_points(ctx, ctx->in_pts.as<float4>(), n, nullptr);
        if (rc) return rc;
        CU(cudaStreamSynchronize(ctx->st));   // (a page-locked `pts` is read asynchronously) the caller may reuse or free it now
        return O3R_OK;
    });
}

int o3r_cloud_size(o3r_ctx* ctx, size_t* n) {
    if (!n) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (ctx->retain()) { *n = ctx->res.n_cloud; return O3R_OK; }
        int rc = refresh_nres(ctx, true);
        if (rc) return rc;
        *n = ctx->res.n_ub;
        return O3R_OK;
    });
}

int o3r_cloud_clear(o3r_ctx* ctx) {
    return api(ctx, [&] {
        CU(cudaStreamSynchronize(ctx->st));
        ctx->rt.reset();
        { int rc = res_clear(ctx); if (rc) return rc; }
        if (ctx->chg) chg_reset(ctx, false);
        return O3R_OK;
    });
}

// engine 1 on an arbitrary device cloud of one segment
static int voxel_grid_dev(o3r_ctx* ctx, const float4* pts, size_t n, float ix, float iy, float iz, uint32_t min_points,
                          int z_shift, float4* out, uint64_t* out_keys, uint32_t* out_counts, size_t* n_out,
                          int* passthrough) {
    if (n >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "cloud too large for 32-bit indices");
    CU(ctx->seg2.ensure(16));
    const uint32_t seg_h[2] = {0u, (uint32_t)n};
    { int rcu = upload_small(ctx, ctx->seg2.p, seg_h, 8); if (rcu) return rcu; }
    const uint32_t* seg = ctx->seg2.as<uint32_t>();
    CU(ctx->bbox.ensure(6 * 4));
    CU(ctx->grids.ensure(sizeof(GridParams)));
    FILL(ctx->bbox.as<uint32_t>(), (size_t)(1) * 24, FILL_BBOX);
    LAUNCH(k_bbox_pts, dim3(cdiv(n, kTileV), 1), kThreads, 0, pts, seg, z_shift, ctx->bbox.as<uint32_t>());
    LAUNCH(k_grid_params, 1, 32, 0, 1, ctx->bbox.as<uint32_t>(), ix, iy, iz, ctx->grids.as<GridParams>());
    int rc = vg_one_segment(ctx, pts, seg, n, ix, iy, iz, min_points, z_shift, out, out_keys, out_counts, n_out);
    if (rc) return rc;
    if (passthrough) {
        GridParams g;
        CU(cudaMemcpyAsync(&g, ctx->grids.p, sizeof(g), cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
        *passthrough = g.passthrough;
    }
    return O3R_OK;
}

// downsamplePtCloud(cloud_big, true) into a device buffer: *res = result, *m = records
// When *exact_pending comes back true, *m is only an upper bound and the exact record count is still on the device
// (cnt[CNT_EMIT]): the caller queues its read-back (and the output copy) behind the kernels and syncs ONCE.
static int cloud_downsample_dev(o3r_ctx* ctx, const float4** res, size_t* m, bool* exact_pending) {
    *res = nullptr; *m = 0;
    if (exact_pending) *exact_pending = false;
    if (ctx->p.dont_downsample) {  // pose.cpp:533-536: cloud_small = cloud_big
        *res = ctx->res.cloud.as<float4>(); *m = ctx->res.n_cloud;
        return O3R_OK;
    }
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    if (ctx->retain() && ctx->comm) return retain_downsample_sharded(ctx, res, m);   // collective (host_retain.cuh)
    if (ctx->retain()) {  // one-shot pcl::VoxelGrid over cloud_big, exactly pose_functions.cpp:1654-1709
        if (ctx->res.n_cloud == 0) return O3R_OK;
        CU(ctx->ckey.ensure(ctx->res.n_cloud * 16));   // result points (<= n_cloud)
        int rc = voxel_grid_dev(ctx, ctx->res.cloud.as<float4>(), ctx->res.n_cloud, ctx->inv_c, ctx->inv_c, ctx->inv_cz,
                                ctx->p.min_points_per_voxel, 1, ctx->ckey.as<float4>(), nullptr, nullptr, m, nullptr);
        if (rc) return rc;
        *res = ctx->ckey.as<float4>();
        return O3R_OK;
    }
    // device-driven: launches are sized by the host's upper bound of the resident count, the kernels read the exact one
    { int rc0 = refresh_nres(ctx, false); if (rc0) return rc0; }
    const size_t n_ub = ctx->res.n_ub;
    if (n_ub == 0) return O3R_OK;
    const ResCells R = res_cells(ctx);
    const uint32_t tiles = cdiv(n_ub, kTileV);
    CU(ctx->new_cnt.ensure((size_t)tiles * 4));
    CU(ctx->new_off.ensure((size_t)tiles * 4));
    CU(ctx->cacc.ensure(n_ub * 16));
    LAUNCH(k_acc_emit_cnt, tiles, kThreads, 0, cnt + CNT_NRES, R.acc, ctx->p.min_points_per_voxel,
           ctx->new_cnt.as<uint32_t>());
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->new_cnt.as<uint32_t>(), ctx->new_off.as<uint32_t>(), tiles, cnt + CNT_EMIT);
    LAUNCH(k_acc_emit, tiles, kThreads, 0, cnt + CNT_NRES, R.acc, R.rgb, ctx->p.min_points_per_voxel, ctx->new_off.as<uint32_t>(), ctx->cacc.as<float4>());
    *res = ctx->cacc.as<float4>();
    *m = n_ub;   // upper bound; the exact count is cnt[CNT_EMIT] once the stream has run (callers read it back)
    if (exact_pending) *exact_pending = true;
    return O3R_OK;
}

// one read-back of the exact output count (and of the resident count, which tightens the host's bound)
static int downsample_finish(o3r_ctx* ctx, size_t* m) {
    { int rc = res_read_back(ctx); if (rc) return rc; }
    *m = ctx->h_counters[CNT_EMIT];
    if (ctx->x.pending_check) {   // the exchanges since the last read-back: did a slot overflow?
        ctx->x.pending_check = false;
        if (ctx->h_counters[CNT_XFLAG]) return x_overflow(ctx);
    }
    return O3R_OK;
}

int o3r_cloud_downsample(o3r_ctx* ctx, o3r_point* out, size_t cap, size_t* n_out) {
    return api(ctx, [&] {
        if (n_out) *n_out = 0;
        const float4* res;
        size_t m;
        bool pending;
        int rc = cloud_downsample_dev(ctx, &res, &m, &pending);
        if (rc) return rc;
        if (!pending) return copy_out(ctx, res, m, out, cap, n_out);
        // accumulators: the copy of up to min(cap, bound) records is queued behind the emit kernels, one sync for everything
        const size_t ncopy = (out && cap) ? std::min(cap, m) : 0;
        if (ncopy) CU(cudaMemcpyAsync(out, res, ncopy * 16, cudaMemcpyDeviceToHost, ctx->st));
        rc = downsample_finish(ctx, &m);
        if (rc) return rc;
        if (n_out) *n_out = m;
        if (!out && cap == 0) return O3R_OK;
        if (cap < m) return ctx->fail(O3R_ERR_CAPACITY, "output buffer too small");
        return O3R_OK;
    });
}

int o3r_cloud_downsample_dev(o3r_ctx* ctx, const o3r_point** dev_out, size_t* n_out) {
    if (!n_out) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        const float4* res;
        bool pending;
        int rc = cloud_downsample_dev(ctx, &res, n_out, &pending);
        if (rc) return rc;
        if (pending) { rc = downsample_finish(ctx, n_out); if (rc) return rc; }
        else CU(cudaStreamSynchronize(ctx->st));
        if (dev_out) *dev_out = reinterpret_cast<const o3r_point*>(res);
        return O3R_OK;
    });
}

int o3r_cloud_track_changes(o3r_ctx* ctx, int enable) {
    return api(ctx, [&] {
        { int rc = chg_check_mode(ctx); if (rc) return rc; }
        if (!enable) {
            CU(cudaStreamSynchronize(ctx->st));   // (queued unions may still read or write the buffers)
            ctx->chg.reset();
            return O3R_OK;
        }
        if (!ctx->chg) ctx->chg.reset(new ChangeTracking());
        chg_reset(ctx, true);   // the next read returns the full state
        return O3R_OK;
    });
}

int o3r_cloud_changes(o3r_ctx* ctx, o3r_point* out, uint64_t* keys, uint32_t* counts, size_t cap, size_t* n_out) {
    if (!n_out) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        *n_out = 0;
        int rc = chg_compute(ctx);
        if (rc) return rc;
        const size_t m = ctx->chg->m;
        *n_out = m;
        if (!out && cap == 0) return O3R_OK;   // size query: nothing consumed
        if (cap < m) return ctx->fail(O3R_ERR_CAPACITY, "output buffer too small");
        if (m) {
            if (out) CU(cudaMemcpyAsync(out, ctx->chg->out.p, m * 16, cudaMemcpyDeviceToHost, ctx->st));
            if (keys) CU(cudaMemcpyAsync(keys, ctx->chg->okeys.p, m * 8, cudaMemcpyDeviceToHost, ctx->st));
            if (counts) CU(cudaMemcpyAsync(counts, ctx->chg->ocnt.p, m * 4, cudaMemcpyDeviceToHost, ctx->st));
            CU(cudaStreamSynchronize(ctx->st));
        }
        chg_reset(ctx, false);   // delivered: nothing is pending any more
        return O3R_OK;
    });
}

int o3r_cloud_changes_dev(o3r_ctx* ctx, const o3r_point** dev_out, const uint64_t** dev_keys, const uint32_t** dev_counts,
                          size_t* n_out) {
    if (!n_out) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        *n_out = 0;
        int rc = chg_compute(ctx);
        if (rc) return rc;
        *n_out = ctx->chg->m;
        if (dev_out) *dev_out = ctx->chg->out.as<const o3r_point>();
        if (dev_keys) *dev_keys = ctx->chg->okeys.as<const uint64_t>();
        if (dev_counts) *dev_counts = ctx->chg->ocnt.as<const uint32_t>();
        chg_reset(ctx, false);   // (the records stay in the context's buffers until the next call)
        return O3R_OK;
    });
}

int o3r_cloud_export_cells(o3r_ctx* ctx, o3r_cell* out, size_t cap, size_t* n_out) {
    if (!n_out) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        *n_out = 0;
        return export_cells_impl(ctx, out, cap, n_out);
    });
}

int o3r_cloud_import_cells(o3r_ctx* ctx, const o3r_cell* cells, size_t n) {
    if (n && !cells) return O3R_ERR_INVALID;
    return api(ctx, [&] { return import_cells_impl(ctx, cells, n); });
}

int o3r_cloud_export_points(o3r_ctx* ctx, o3r_point* out, size_t cap, size_t* n_out) {
    if (!n_out) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        *n_out = 0;
        return export_points_impl(ctx, out, cap, n_out);
    });
}

int o3r_cloud_register(o3r_ctx* ctx, const o3r_point* pts, size_t n, const float T_init[16], const o3r_register_params* params,
                       float T_out[16], o3r_register_stats* stats) {
    if ((n && !pts) || !T_init || !T_out) return O3R_ERR_INVALID;
    return api(ctx, [&] { return register_impl(ctx, pts, true, n, T_init, params, T_out, stats); });
}

int o3r_cloud_register_dev(o3r_ctx* ctx, const o3r_point* dev_pts, size_t n, const float T_init[16],
                           const o3r_register_params* params, float T_out[16], o3r_register_stats* stats) {
    if ((n && !dev_pts) || !T_init || !T_out) return O3R_ERR_INVALID;
    return api(ctx, [&] { return register_impl(ctx, dev_pts, false, n, T_init, params, T_out, stats); });
}

int o3r_cloud_mesh(o3r_ctx* ctx, double max_step, o3r_point* verts, float* normals, size_t vcap, size_t* n_verts,
                   uint32_t* tris, size_t tcap, size_t* n_tris) {
    if (!n_verts || !n_tris) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        const MeshOut out{verts, normals, vcap, tris, tcap};
        return mesh_impl(ctx, max_step, &out, n_verts, n_tris);
    });
}

int o3r_cloud_mesh_dev(o3r_ctx* ctx, double max_step, const o3r_point** verts, const float** normals, size_t* n_verts,
                       const uint32_t** tris, size_t* n_tris) {
    if (!n_verts || !n_tris) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (verts) *verts = nullptr;
        if (normals) *normals = nullptr;
        if (tris) *tris = nullptr;
        const int rc = mesh_impl(ctx, max_step, nullptr, n_verts, n_tris);
        if (rc) return rc;
        if (verts) *verts = ctx->mesh.verts.as<const o3r_point>();
        if (normals) *normals = ctx->mesh.normals.as<const float>();
        if (tris) *tris = ctx->mesh.tris.as<const uint32_t>();
        return O3R_OK;
    });
}

int o3r_voxel_grid(o3r_ctx* ctx, const o3r_point* pts, size_t n, float lx, float ly, float lz, unsigned min_points,
                   o3r_point* out, size_t cap, size_t* n_out, uint64_t* keys, uint32_t* counts, int* passthrough) {
    if (!n_out || (n && !pts)) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        *n_out = 0;
        if (passthrough) *passthrough = 0;
        if (n == 0) return O3R_OK;
        if (!(lx > 0) || !(ly > 0) || !(lz > 0)) return ctx->fail(O3R_ERR_INVALID, "leaf size must be positive");
        CU(ctx->in_pts.ensure(n * 16));
        CU(ctx->out_pts.ensure(n * 16));
        CU(ctx->ckey.ensure(n * 8));
        CU(ctx->new_keys.ensure(n * 4));
        CU(cudaMemcpyAsync(ctx->in_pts.p, pts, n * 16, cudaMemcpyHostToDevice, ctx->st));
        size_t m = 0;
        int rc = voxel_grid_dev(ctx, ctx->in_pts.as<float4>(), n, 1.0f / lx, 1.0f / ly, 1.0f / lz, min_points, 0,
                                ctx->out_pts.as<float4>(), ctx->ckey.as<uint64_t>(), ctx->new_keys.as<uint32_t>(), &m, passthrough);
        if (rc) return rc;
        *n_out = m;
        if (!out && cap == 0) return O3R_OK;
        if (cap < m) return ctx->fail(O3R_ERR_CAPACITY, "output buffer too small");
        if (m) {
            CU(cudaMemcpyAsync(out, ctx->out_pts.p, m * 16, cudaMemcpyDeviceToHost, ctx->st));
            if (keys) CU(cudaMemcpyAsync(keys, ctx->ckey.p, m * 8, cudaMemcpyDeviceToHost, ctx->st));
            if (counts) CU(cudaMemcpyAsync(counts, ctx->new_keys.p, m * 4, cudaMemcpyDeviceToHost, ctx->st));
            CU(cudaStreamSynchronize(ctx->st));
        }
        return O3R_OK;
    });
}

int o3r_blur_u8(o3r_ctx* ctx, const uint8_t* src, size_t src_step, int rows, int cols, int kernel, int mode,
                uint8_t* dst, size_t dst_step) {
    if (!src || !dst || rows <= 0 || cols <= 0) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (kernel < 1 || kernel > kBlurMaxK) return ctx->fail(O3R_ERR_INVALID, "kernel must be in 1..127");
        if (mode == O3R_BLUR_MEDIAN && (kernel & 1) == 0)
            return ctx->fail(O3R_ERR_INVALID, "median blur needs an odd kernel (cv::medianBlur asserts)");
        if (mode != O3R_BLUR_MEDIAN && mode != O3R_BLUR_BOX && mode != O3R_BLUR_BILATERAL)
            return ctx->fail(O3R_ERR_INVALID, "unknown blur mode");
        const size_t step = ((size_t)cols + 15) & ~(size_t)15, plane = step * rows;
        CU(ctx->blur.disp.ensure(plane));
        CU(ctx->blur.out.ensure(plane));
        CU(ctx->blur.jobs.ensure(sizeof(BlurJob)));
        CU(cudaMemcpy2DAsync(ctx->blur.disp.p, step, src, src_step, cols, rows, cudaMemcpyHostToDevice, ctx->st));
        BlurJob job{ctx->blur.disp.as<uint8_t>(), step, ctx->blur.out.as<uint8_t>(), step};
        CU(cudaMemcpyAsync(ctx->blur.jobs.p, &job, sizeof(job), cudaMemcpyHostToDevice, ctx->st));
        const dim3 g(cdiv(cols, kBlurStrip), cdiv(rows, blur_rows(mode)), 1);
        const size_t sm = blur_smem(kernel, mode);
        if (mode == O3R_BLUR_BILATERAL) {
            BilateralLut L;
            int rcl = bilateral_lut(ctx, kernel, &L);
            if (rcl) return rcl;
            const dim3 gb(cdiv(cols, kBilW), cdiv(rows, kBilTY), 1);
            LAUNCH(k_bilateral, gb, dim3(kBilTX, kBilTY), bilateral_smem(L.radius, L.maxk), ctx->blur.jobs.as<BlurJob>(), L, rows, cols, 0, 0, cols, rows);
        } else if (mode == O3R_BLUR_MEDIAN)
            LAUNCH_N("k_blur_median", (k_blur<O3R_BLUR_MEDIAN>), g, kBlurRows, sm, ctx->blur.jobs.as<BlurJob>(), rows, cols, kernel, 0, 0, cols, rows);
        else
            LAUNCH_N("k_blur_box", (k_blur<O3R_BLUR_BOX>), g, kBlurRows, sm, ctx->blur.jobs.as<BlurJob>(), rows, cols, kernel, 0, 0, cols, rows);
        CU(cudaMemcpy2DAsync(dst, dst_step, ctx->blur.out.p, step, cols, rows, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
        return O3R_OK;
    });
}

// ---- the exchange inside the library: communicator + one call per cycle (SURVEY 8e) --------------------------------------
int o3r_comm_unique_id(void* id_out) {
    if (!id_out) return O3R_ERR_INVALID;
    NcclApi* N = nccl_api();
    if (!N->err.empty()) { g_create_err = N->err; return O3R_ERR_CUDA; }
    ncclUniqueId id;
    if (N->GetUniqueId(&id) != ncclSuccess) { g_create_err = "ncclGetUniqueId failed"; return O3R_ERR_CUDA; }
    memcpy(id_out, &id, sizeof(id));
    return O3R_OK;
}

int o3r_comm_init(o3r_ctx* ctx, int world, int rank, const void* id, size_t slot_cells) {
    if (!id) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        NcclApi* N = nccl_api();
        if (!N->err.empty()) return ctx->fail(O3R_ERR_CUDA, N->err);
        if (ctx->comm) return ctx->fail(O3R_ERR_INVALID, "the context already has a communicator");
        int rc = comm_setup(ctx, world, rank, slot_cells);
        if (rc) return rc;
        ZERO(ctx->counters.as<uint32_t>() + CNT_XFLAG, 8);
        ncclUniqueId uid;
        memcpy(&uid, id, sizeof(uid));
        ncclComm_t c = nullptr;
        NC(N->CommInitRank(&c, world, uid, rank));
        ctx->comm = c; ctx->comm_owned = true;
        return O3R_OK;
    });
}

int o3r_comm_attach(o3r_ctx* ctx, void* nccl_comm, int world, int rank, size_t slot_cells) {
    if (!nccl_comm) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        NcclApi* N = nccl_api();
        if (!N->err.empty()) return ctx->fail(O3R_ERR_CUDA, N->err);
        if (ctx->comm) return ctx->fail(O3R_ERR_INVALID, "the context already has a communicator");
        int rc = comm_setup(ctx, world, rank, slot_cells);
        if (rc) return rc;
        ZERO(ctx->counters.as<uint32_t>() + CNT_XFLAG, 8);
        ctx->comm = nccl_comm; ctx->comm_owned = false;
        return O3R_OK;
    });
}

int o3r_comm_destroy(o3r_ctx* ctx) {
    return api(ctx, [&] {
        CU(cudaStreamSynchronize(ctx->st));
        NcclApi* N = nccl_api();
        if (ctx->comm && ctx->comm_owned) NC(N->CommDestroy((ncclComm_t)ctx->comm));
        ctx->comm = nullptr; ctx->comm_owned = false; ctx->world = 1; ctx->rank = 0;
        ctx->x = Exchange();
        ctx->rt = RetainShard();
        return O3R_OK;
    });
}

int o3r_exchange_cycle(o3r_ctx* ctx) {
    return api(ctx, [&] {
        if (ctx->comm && ctx->retain()) return O3R_OK;   // RETAIN: the points stay where they were made; o3r_cloud_downsample exchanges
        return exchange_cycle_impl(ctx);
    });
}

// ---- pre-pass (SURVEY §8f-3) ---------------------------------------------------------------------------------------------
namespace {

// symmetric 3x3 eigen-decomposition by cyclic Jacobi rotations: AtA = V diag(w) V^T (what cv::invert(AtA, DECOMP_SVD)
// needs for a symmetric positive semi-definite matrix)
void sym3_eigen(double A[3][3], double V[3][3], double w[3]) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) V[i][j] = (i == j);
    for (int sweep = 0; sweep < 64; ++sweep) {
        const double off = std::fabs(A[0][1]) + std::fabs(A[0][2]) + std::fabs(A[1][2]);
        if (off == 0.0) break;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                if (A[p][q] == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
                for (int k = 0; k < 3; ++k) {
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - sn * akq;
                    A[k][q] = sn * akp + c * akq;
                }
                for (int k = 0; k < 3; ++k) {
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - sn * aqk;
                    A[q][k] = sn * apk + c * aqk;
                }
                for (int k = 0; k < 3; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - sn * vkq;
                    V[k][q] = sn * vkp + c * vkq;
                }
            }
    }
    for (int i = 0; i < 3; ++i) w[i] = A[i][i];
}

// getMean + getVariance (pose_functions.cpp:987-1028) of the ROI; the sample source is already on the device
int roi_variance(o3r_ctx* ctx, const uint8_t* d_disp, size_t dstep, const uint8_t* d_labels, size_t lstep,
                 const double* d_coef, int n_planes, double* variance) {
    const o3r_params& p = ctx->p;
    const int nrow = p.rows - 2 * p.bounding_box, ncol = p.cols - p.bounding_box - p.cols_start_aft_cutout;
    if (nrow <= 0 || ncol <= 0) return ctx->fail(O3R_ERR_INVALID, "empty ROI");
    CU(ctx->pp.rows.ensure((size_t)nrow * 8));
    std::vector<double> rows_h(nrow);
    double mean = 0.0;
    for (int pass = 0; pass < 2; ++pass) {
        LAUNCH(k_row_moment, nrow, kThreads, 0, d_disp, dstep, d_labels, lstep, d_coef, n_planes, p.cols,
               p.cols_start_aft_cutout, p.bounding_box, p.min_disparity, pass, mean, ctx->pp.rows.as<double>());
        CU(cudaMemcpyAsync(rows_h.data(), ctx->pp.rows.p, (size_t)nrow * 8, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
        double s = 0.0;
        for (int r = 0; r < nrow; ++r) s += rows_h[r];
        if (pass == 0) mean = s / ((double)nrow * ncol);            // :1004 (divides by ALL ROI pixels)
        else *variance = s / ((double)nrow * ncol - 1);             // :1026
    }
    return O3R_OK;
}

int stage_plane_u8(o3r_ctx* ctx, DevBuf& buf, const uint8_t* src, size_t src_step, size_t* step_out) {
    const o3r_params& p = ctx->p;
    const size_t step = ((size_t)p.cols + 15) & ~(size_t)15;
    CU(buf.ensure(step * p.rows));
    CU(cudaMemcpy2DAsync(buf.p, step, src, src_step, p.cols, p.rows, cudaMemcpyHostToDevice, ctx->st));
    *step_out = step;
    return O3R_OK;
}

}  // namespace

int o3r_disp_variance(o3r_ctx* ctx, const uint8_t* disp, size_t disp_step, double* variance) {
    if (!disp || !variance) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        size_t step;
        int rc = stage_plane_u8(ctx, ctx->pp.disp, disp, disp_step, &step);
        if (rc) return rc;
        return roi_variance(ctx, ctx->pp.disp.as<uint8_t>(), step, nullptr, 0, nullptr, 0, variance);
    });
}

int o3r_plane_fit(o3r_ctx* ctx, const uint8_t* labels, size_t labels_step, const uint8_t* disp, size_t disp_step,
                  double* coef, int coef_cap, int* n_planes, double* variance) {
    if (!labels || !disp || !coef || !n_planes) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        const o3r_params& p = ctx->p;
        size_t lstep, dstep;
        int rc = stage_plane_u8(ctx, ctx->pp.labels, labels, labels_step, &lstep);
        if (rc) return rc;
        rc = stage_plane_u8(ctx, ctx->pp.disp, disp, disp_step, &dstep);
        if (rc) return rc;
        const size_t sum_bytes = (size_t)256 * kLabSums * 8;
        CU(ctx->pp.sums.ensure(sum_bytes));
        ZERO(ctx->pp.sums.p, sum_bytes);
        LAUNCH(k_label_sums, cdiv(p.rows, 8), kThreads, 0, ctx->pp.labels.as<uint8_t>(), lstep, ctx->pp.disp.as<uint8_t>(), dstep,
               p.rows, p.cols, p.cols_start_aft_cutout, p.bounding_box, ctx->pp.sums.as<unsigned long long>());
        std::vector<unsigned long long> S((size_t)256 * kLabSums);
        CU(cudaMemcpyAsync(S.data(), ctx->pp.sums.p, sum_bytes, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
        int np = 0;
        for (int cluster = 1; cluster < 256; ++cluster) {   // :907 (labels are 8-bit); stops at the first absent label (:923)
            const unsigned long long* s = &S[(size_t)cluster * kLabSums];
            if (s[0] == 0) break;
            if (cluster > coef_cap) return ctx->fail(O3R_ERR_CAPACITY, "coef buffer too small");
            double* c = coef + 3 * (cluster - 1);
            c[0] = c[1] = c[2] = 0.0;
            np = cluster;
            if (s[1] == 0) continue;   // :939-940: no pixel inside the ROI, the label keeps 0.0
            // :957-965: x = inv_SVD(AtA) * At * b with AtA = [[Sxx Sxy Sx][Sxy Syy Sy][Sx Sy n]], At*b = [Sxd Syd Sd]
            double A[3][3] = {{(double)s[4], (double)s[5], (double)s[2]}, {(double)s[5], (double)s[6], (double)s[3]},
                              {(double)s[2], (double)s[3], (double)s[1]}};
            double V[3][3], w[3];
            sym3_eigen(A, V, w);
            const double thr = DBL_EPSILON * 2 * (std::fabs(w[0]) + std::fabs(w[1]) + std::fabs(w[2]));
            const double rhs[3] = {(double)s[7], (double)s[8], (double)s[9]};
            for (int i = 0; i < 3; ++i) {
                double acc = 0;
                for (int j = 0; j < 3; ++j) {
                    double inv_ij = 0;
                    for (int e = 0; e < 3; ++e)
                        if (std::fabs(w[e]) > thr) inv_ij += V[i][e] * V[j][e] / w[e];
                    acc += inv_ij * rhs[j];
                }
                c[i] = acc;
            }
        }
        *n_planes = np;
        if (variance) {   // getVariance(new_disp_img, true), :973; the caller applies the > 3 gate (:975-982)
            CU(ctx->pp.coef.ensure(std::max(np, 1) * 24));
            if (np) { int rcu = upload_small(ctx, ctx->pp.coef.p, coef, (size_t)np * 24); if (rcu) return rcu; }
            return roi_variance(ctx, nullptr, 0, ctx->pp.labels.as<uint8_t>(), lstep, ctx->pp.coef.as<double>(), np, variance);
        }
        return O3R_OK;
    });
}


int o3r_sor(o3r_ctx* ctx, const o3r_point* pts, size_t n, int mean_k, double stddev_mul, uint8_t* keep, float* dist,
            double* threshold) {
    if ((n && !pts) || !keep) return O3R_ERR_INVALID;
    return api(ctx, [&] {
        if (n == 0) return O3R_OK;
        if (n >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "cloud too large for 32-bit indices");
        CU(ctx->in_pts.ensure(n * 16));
        CU(ctx->seg2.ensure(16));
        CU(cudaMemcpyAsync(ctx->in_pts.p, pts, n * 16, cudaMemcpyHostToDevice, ctx->st));
        const uint32_t seg_h[2] = {0u, (uint32_t)n};
        { int rcu = upload_small(ctx, ctx->seg2.p, seg_h, 8); if (rcu) return rcu; }
        SortU32 sb;
        int rc = carve_sort_u32(ctx, n, sb);
        if (rc) return rc;
        rc = sor_filter(ctx, sb, ctx->in_pts.as<float4>(), ctx->seg2.as<uint32_t>(), 1, n, mean_k, stddev_mul);
        if (rc) return rc;
        std::vector<float> d(n);
        double thr = 0;
        CU(cudaMemcpyAsync(d.data(), ctx->sor.dist.p, n * 4, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaMemcpyAsync(&thr, ctx->sor.thr.p, 8, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
        for (size_t i = 0; i < n; ++i) keep[i] = !((double)d[i] > thr);
        if (dist) memcpy(dist, d.data(), n * 4);
        if (threshold) *threshold = thr;
        return O3R_OK;
    });
}

}  // extern "C"
