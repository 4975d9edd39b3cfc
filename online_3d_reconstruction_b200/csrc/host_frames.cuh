// host_frames.cuh — the batched per-frame path: input staging / prefetch, stage A, SOR, per-frame VoxelGrid, tile pre-reduction, merge
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "host_merge.cuh"
#include "host_sor.cuh"
#include "host_bucket.cuh"
#include "host_tile.cuh"

namespace {

// ---- the batched per-frame path ------------------------------------------------------------------------------------
struct BatchOpts {
    bool merge = true;          // append / merge into the resident cloud
    uint8_t* mask_dev = nullptr;  // optional validity mask output
    bool mask_only = false;
};

// stage A for one chunk of frames (descriptors at `fr`).  V1 mode: points + leaf indices into the chunk scratch.
// dont_downsample mode: points straight into the batch buffer at the device-side running offset.
template <int DT>
int launch_stage_a(o3r_ctx* ctx, const AParams& P, const FrameDev* fr, int n, const BatchOpts& opt, float4* pts_out,
                   uint32_t* keys_out, const uint32_t* out_base, uint32_t* goff) {
    const dim3 grid(P.tiles_per_frame, n);
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    FILL(ctx->bbox.as<uint32_t>(), (size_t)(n) * 24, FILL_BBOX);
    LAUNCH_N("k_pre", (k_pre<DT>), grid, kThreads, 0, P, fr, ctx->tile_cnt.as<uint32_t>(), ctx->bbox.as<uint32_t>(),
             opt.mask_dev);
    if (opt.mask_only) return O3R_OK;
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, ctx->tile_cnt.as<uint32_t>(), ctx->tile_off.as<uint32_t>(),
           (uint32_t)((size_t)P.tiles_per_frame * n), cnt + CNT_PTS);
    LAUNCH(k_a_post, cdiv(n + 1, kThreads), kThreads, 0, n, P.tiles_per_frame, ctx->tile_off.as<uint32_t>(),
           cnt + CNT_PTS, ctx->bbox.as<uint32_t>(), ctx->inv_f, ctx->inv_f, ctx->inv_f, P.want_keys,
           ctx->frame_off.as<uint32_t>(), ctx->grids.as<GridParams>(), out_base, goff);
    LAUNCH_N("k_emit", (k_emit<DT>), grid, kThreads, 0, P, fr, ctx->tile_off.as<uint32_t>(),
             ctx->frame_off.as<uint32_t>(), ctx->grids.as<GridParams>(), pts_out, keys_out, out_base);
    return O3R_OK;
}

// ---- input staging (host entry points) --------------------------------------------------------------------------------
struct StageGeom { size_t es, dstep, dplane, cstep, cplane, lstep, lplane; };

StageGeom stage_geom(const o3r_params& p, int disp_type) {
    StageGeom G;
    G.es = disp_elem(disp_type);
    G.dstep = (((size_t)p.cols * G.es) + 15) & ~(size_t)15; G.dplane = G.dstep * p.rows;
    G.cstep = (((size_t)p.cols * 3) + 15) & ~(size_t)15;     G.cplane = G.cstep * p.rows;
    G.lstep = ((size_t)p.cols + 15) & ~(size_t)15;           G.lplane = G.lstep * p.rows;
    return G;
}

void frames_signature(const o3r_frame* frames, int n, std::vector<const void*>& sig) {
    sig.clear();
    sig.reserve((size_t)n * 4);
    for (int i = 0; i < n; ++i) {
        sig.push_back(frames[i].disp); sig.push_back(frames[i].bgr);
        sig.push_back(frames[i].labels); sig.push_back(frames[i].kp_xy);
    }
}

// sizes staging set `set` for the frames and fills their device-side descriptors (everything but T)
int stage_layout(o3r_ctx* ctx, const o3r_frame* frames, int n, bool label_mode, int J, const StageGeom& G, int set,
                 std::vector<FrameDev>& fd) {
    o3r_ctx::Staging& S = ctx->stg[set];
    size_t kp_total = 0, coef_total = 0;
    for (int i = 0; i < n; ++i) {
        const o3r_frame& f = frames[i];
        kp_total += (J != 1 && f.kp_xy && f.n_kp > 0) ? (size_t)f.n_kp * 2 : 0;
        coef_total += label_mode ? (size_t)std::max(f.n_planes, 0) * 3 : 0;
    }
    if (!label_mode) CU(S.disp.ensure(G.dplane * n));
    CU(S.bgr.ensure(G.cplane * n));
    if (label_mode) { CU(S.labels.ensure(G.lplane * n)); CU(S.coef.ensure(std::max<size_t>(coef_total, 1) * 8)); }
    if (kp_total) CU(S.kp.ensure(kp_total * 4));
    size_t kp_at = 0, coef_at = 0;
    for (int i = 0; i < n; ++i) {
        const o3r_frame& f = frames[i];
        FrameDev& d = fd[i];
        const int nk = (J != 1 && f.kp_xy && f.n_kp > 0) ? f.n_kp : 0;
        d.disp = label_mode ? nullptr : S.disp.as<uint8_t>() + G.dplane * i; d.disp_step = G.dstep;
        d.bgr = S.bgr.as<uint8_t>() + G.cplane * i; d.bgr_step = G.cstep;
        d.labels = label_mode ? S.labels.as<uint8_t>() + G.lplane * i : nullptr; d.labels_step = G.lstep;
        d.plane_coef = label_mode ? S.coef.as<double>() + coef_at : nullptr;
        d.kp_xy = nk ? S.kp.as<float>() + kp_at : nullptr;
        d.n_planes = label_mode ? std::max(f.n_planes, 0) : 0;
        d.n_kp = nk;
        kp_at += (size_t)nk * 2; coef_at += (size_t)d.n_planes * 3;
    }
    return O3R_OK;
}

// issues the H2D copies of frames [f0, f0 + nc): groups of frames alternate between the two copy streams, and the first stream
// then waits for the second, so an event recorded on st_copy after this call covers every copy
int stage_copy(o3r_ctx* ctx, const o3r_frame* frames, const std::vector<FrameDev>& fd, int f0, int nc, bool label_mode,
               const StageGeom& G) {
    const o3r_params& p = ctx->p;
    // Only the pixels the path can read cross PCIe: the scan ROI x in [x0, cols-bb), y in [bb, rows-bb)
    // (pose_functions.cpp:1062,1094-1095; keypoints outside it are rejected too), widened by the blur window's reach for
    // the disparity plane.  The device planes keep the full-image layout, so the kernels index as before.
    const int halo = p.blur_kernel > 1 ? p.blur_kernel / 2 + 1 : 0;
    const int cx0 = std::min(p.cols, std::max(0, p.cols_start_aft_cutout)), cx1 = std::max(cx0, p.cols - p.bounding_box);
    const int cy0 = std::min(p.rows, std::max(0, p.bounding_box)), cy1 = std::max(cy0, p.rows - p.bounding_box);
    const int dx0 = std::max(0, cx0 - halo), dx1 = std::min(p.cols, cx1 + halo);
    const int dy0 = std::max(0, cy0 - halo), dy1 = std::min(p.rows, cy1 + halo);
    if (cx1 <= cx0 || cy1 <= cy0) return O3R_OK;   // empty ROI: nothing is ever read
    // Frames whose planes sit back to back in host memory (a cycle held in one pinned arena, same row pitch) move as ONE 3-D
    // copy per plane type and group: the group's planes form a pitched volume on both sides (the staging planes are back to
    // back as well) whose extent (ROI bytes per row, ROI rows, frames) is exactly the ROIs.  Measured on B200
    // (profiles/scripts/h2d_shapes.py, 50-frame 720p cycle): 100 per-plane 2-D copies 3.21 ms (each costs ~5 us of set-up on the
    // engine), one 2-D copy per plane type with the margin rows between the ROIs riding along 2.97 ms, one 3-D copy 2.81 ms.
    const int kGroup = 16;
    int gi = 0;
    for (int i = f0; i < f0 + nc; ++gi) {
        int j = i + 1;
        if (!label_mode)
            while (j < f0 + nc && j - i < kGroup && frames[j].disp_step == frames[i].disp_step && frames[j].bgr_step == frames[i].bgr_step &&
                   (const uint8_t*)frames[j].disp == (const uint8_t*)frames[j - 1].disp + (size_t)p.rows * frames[i].disp_step &&
                   frames[j].bgr == frames[j - 1].bgr + (size_t)p.rows * frames[i].bgr_step &&
                   (const uint8_t*)fd[j].disp == (const uint8_t*)fd[j - 1].disp + G.dplane && fd[j].bgr == fd[j - 1].bgr + G.cplane)
                ++j;
        const o3r_frame& f = frames[i];
        const FrameDev& d = fd[i];
        cudaStream_t cs = (gi & 1) ? ctx->st_copy2 : ctx->st_copy;
        if (j - i > 1) {   // a group: ONE 3-D copy per plane type, extent (ROI bytes per row, ROI rows, frames) — exactly the ROIs
            auto copy3d = [&](const void* src, size_t spitch, void* dst, size_t dpitch, size_t xb, size_t wb, int y0, int h) {
                cudaMemcpy3DParms q;
                memset(&q, 0, sizeof(q));
                q.srcPtr = make_cudaPitchedPtr(const_cast<void*>(src), spitch, spitch, (size_t)p.rows);
                q.dstPtr = make_cudaPitchedPtr(dst, dpitch, dpitch, (size_t)p.rows);
                q.srcPos = make_cudaPos(xb, (size_t)y0, 0);
                q.dstPos = make_cudaPos(xb, (size_t)y0, 0);
                q.extent = make_cudaExtent(wb, (size_t)h, (size_t)(j - i));
                q.kind = cudaMemcpyHostToDevice;
                return cudaMemcpy3DAsync(&q, cs);
            };
            CU(copy3d(f.disp, f.disp_step, (void*)d.disp, G.dstep, (size_t)dx0 * G.es, (size_t)(dx1 - dx0) * G.es, dy0, dy1 - dy0));
            CU(copy3d(f.bgr, f.bgr_step, (void*)d.bgr, G.cstep, (size_t)cx0 * 3, (size_t)(cx1 - cx0) * 3, cy0, cy1 - cy0));
            for (int q = i; q < j; ++q)
                if (fd[q].n_kp) CU(cudaMemcpyAsync((void*)fd[q].kp_xy, frames[q].kp_xy, (size_t)fd[q].n_kp * 8, cudaMemcpyHostToDevice, cs));
            i = j;
            continue;
        }
        if (!label_mode) {
            CU(cudaMemcpy2DAsync((uint8_t*)d.disp + (size_t)dy0 * G.dstep + (size_t)dx0 * G.es, G.dstep,
                                 (const uint8_t*)f.disp + (size_t)dy0 * f.disp_step + (size_t)dx0 * G.es, f.disp_step,
                                 (size_t)(dx1 - dx0) * G.es, dy1 - dy0, cudaMemcpyHostToDevice, cs));
        } else {
            CU(cudaMemcpy2DAsync((uint8_t*)d.labels + (size_t)cy0 * G.lstep + cx0, G.lstep,
                                 f.labels + (size_t)cy0 * f.labels_step + cx0, f.labels_step, (size_t)(cx1 - cx0), cy1 - cy0,
                                 cudaMemcpyHostToDevice, cs));
            if (d.n_planes)
                CU(cudaMemcpyAsync((void*)d.plane_coef, f.plane_coef, (size_t)d.n_planes * 24, cudaMemcpyHostToDevice, cs));
        }
        CU(cudaMemcpy2DAsync((uint8_t*)d.bgr + (size_t)cy0 * G.cstep + (size_t)cx0 * 3, G.cstep,
                             f.bgr + (size_t)cy0 * f.bgr_step + (size_t)cx0 * 3, f.bgr_step, (size_t)(cx1 - cx0) * 3,
                             cy1 - cy0, cudaMemcpyHostToDevice, cs));
        for (int q = i; q < j; ++q)
            if (fd[q].n_kp) CU(cudaMemcpyAsync((void*)fd[q].kp_xy, frames[q].kp_xy, (size_t)fd[q].n_kp * 8, cudaMemcpyHostToDevice, cs));
        i = j;
    }
    if (nc > 1) {
        CU(cudaEventRecord(ctx->ev_copy2, ctx->st_copy2));
        CU(cudaStreamWaitEvent(ctx->st_copy, ctx->ev_copy2, 0));
    }
    return O3R_OK;
}

// issues the copies of a recorded prefetch request into a free staging set
int flush_deferred_prefetch(o3r_ctx* ctx) {
    if (!ctx->deferred.pending) return O3R_OK;
    ctx->deferred.pending = false;
    const o3r_params& p = ctx->p;
    const o3r_frame* frames = ctx->deferred.frames.data();
    const int n = (int)ctx->deferred.frames.size(), disp_type = ctx->deferred.disp_type;
    const bool label_mode = p.use_segment_labels && frames[0].labels && frames[0].plane_coef;
    const StageGeom G = stage_geom(p, disp_type);
    const int set = ctx->free_stage_set();
    o3r_ctx::Prefetch& pf = ctx->prefetch[set];
    pf.valid = false;
    std::vector<FrameDev> fd(n);
    int rc = stage_layout(ctx, frames, n, label_mode, p.jump_pixels, G, set, fd);
    if (rc) return rc;
    rc = stage_copy(ctx, frames, fd, 0, n, label_mode, G);
    if (rc) return rc;
    if (!pf.ev) CU(cudaEventCreateWithFlags(&pf.ev, cudaEventDisableTiming));
    CU(cudaEventRecord(pf.ev, ctx->st_copy));
    frames_signature(frames, n, pf.sig);
    pf.n = n; pf.disp_type = disp_type; pf.seq = ++ctx->prefetch_seq; pf.valid = true;
    return O3R_OK;
}

// the O3R_TRACE line of a FUSED batch: the engine it starts with and the context state that chose it
void trace_fused_engine(const o3r_ctx* ctx, Engine e, const AParams& P, const BatchOpts& opt) {
    fprintf(stderr, "[o3r trace] fused: engine %s (want_keys %d merge %d tile_off %d bucket_off %d canon %d vec %d R %d)\n",
            e == Engine::TILE ? "tile" : e == Engine::BUCKET ? "bucket" : "sort", P.want_keys, (int)opt.merge, (int)ctx->tv_off,
            (int)ctx->bucket_off, ctx->canon, P.vec, ctx->tv_R);
}

// The batched per-frame path.  `frames` hold host pointers (host_inputs: every frame is copied to device staging
// on the copy stream, chunk by chunk, overlapping the previous chunk's kernels) or device pointers.
int frames_cloud_impl(o3r_ctx* ctx, const o3r_frame* frames, int n, int disp_type, uint32_t* frame_counts,
                      const BatchOpts& opt, bool host_inputs) {
    const o3r_params& p = ctx->p;
    const bool trace = trace_on();
    ctx->busy_set = -1;
    const double tr0 = now_ms();
    // sharded RETAIN: every call is one cycle of the order tag, whatever it holds (n = 0: this rank has no frame in it)
    const bool rt_shard = opt.merge && ctx->comm && ctx->retain();
    const uint32_t rt_cycle = ctx->rt_cycles;
    if (rt_shard) { ++ctx->rt_cycles; ctx->rt_valid = false; }
    if (n <= 0) { ctx->last_n = 0; ctx->last_total = 0; return O3R_OK; }
    if (n > 65535) return ctx->fail(O3R_ERR_INVALID, "too many frames in one batch");
    if (disp_type < 0 || disp_type > 3) return ctx->fail(O3R_ERR_INVALID, "bad disp_type");
    const bool label_mode = p.use_segment_labels && frames[0].labels && frames[0].plane_coef;
    if (p.use_segment_labels && !label_mode && disp_type != O3R_DISP_F64)
        return ctx->fail(O3R_ERR_INVALID, "use_segment_labels needs an F64 disparity plane or labels + plane_coef");
    const bool blur = p.blur_kernel > 1;
    if (blur) {  // cv::bilateralFilter / medianBlur reject CV_64F: the reference throws and yields an empty cloud
        if (disp_type != O3R_DISP_U8 || p.use_segment_labels)
            return ctx->fail(O3R_ERR_INVALID, "blur_kernel > 1 requires u8 disparity (OpenCV rejects CV_64F)");
        if (p.blur_mode == O3R_BLUR_MEDIAN && (p.blur_kernel & 1) == 0)
            return ctx->fail(O3R_ERR_INVALID, "median blur needs an odd blur_kernel (cv::medianBlur asserts)");
        if (p.blur_mode != O3R_BLUR_MEDIAN && p.blur_mode != O3R_BLUR_BOX && p.blur_mode != O3R_BLUR_BILATERAL)
            return ctx->fail(O3R_ERR_INVALID, "unknown blur_mode");
        if (p.blur_kernel > kBlurMaxK) return ctx->fail(O3R_ERR_INVALID, "blur_kernel too large (max 127)");
    }
    const int J = p.jump_pixels;
    int max_kp = 0;
    size_t kp_total = 0, coef_total = 0;
    for (int i = 0; i < n; ++i) {
        const o3r_frame& f = frames[i];
        if (!f.bgr || (!f.disp && !label_mode)) return ctx->fail(O3R_ERR_INVALID, "frame without disparity/colour");
        if (label_mode && (!f.labels || !f.plane_coef)) return ctx->fail(O3R_ERR_INVALID, "frame without labels");
        const int nk = (J != 1 && f.kp_xy && f.n_kp > 0) ? f.n_kp : 0;
        max_kp = std::max(max_kp, nk);
        kp_total += (size_t)nk * 2;
        coef_total += label_mode ? (size_t)std::max(f.n_planes, 0) * 3 : 0;
    }

    AParams P;
    memset(&P, 0, sizeof(P));
    P.rows = p.rows; P.cols = p.cols; P.x0 = p.cols_start_aft_cutout; P.bb = p.bounding_box; P.J = J;
    P.nx = ctx->nx; P.ny = ctx->ny; P.npix = ctx->npix;
    P.kp_tiles = (int)cdiv((size_t)max_kp, kTileA);
    P.tiles_per_frame = P.kp_tiles + (int)cdiv(P.npix, kTileA);
    P.label_mode = label_mode;
    P.canon = ctx->canon;
    P.use_lut = ctx->canon && disp_type == O3R_DISP_U8 && !label_mode;
    P.thr_i = (int)std::floor(p.min_disparity);
    P.min_disp = p.min_disparity; P.div = p.disp_divisor;
    for (int i = 0; i < 16; ++i) P.q[i] = p.Q[i];
    P.lut_r = ctx->lut_r.as<double>(); P.lut_z = ctx->lut_z.as<float>();
    P.want_keys = !p.dont_downsample && !opt.mask_only;
    P.want_bbox = P.want_keys;
    if (P.tiles_per_frame == 0) {  // nothing to scan (J == 0 and no keypoints)
        ctx->last_n = n; ctx->last_total = 0; ctx->last_off.assign(n + 1, 0);
        if (frame_counts) std::fill(frame_counts, frame_counts + n, 0u);
        return O3R_OK;
    }

    // ---- device copies of the inputs (host entry points) and frame descriptors
    const size_t es = disp_elem(disp_type);
    const StageGeom G = stage_geom(p, disp_type);
    const size_t blur_step = G.lstep;
    // inputs already on their way (o3r_frames_prefetch of exactly these frames)?
    bool prefetched = false;
    int set = 0;
    if (host_inputs) {
        std::vector<const void*> sig;
        frames_signature(frames, n, sig);
        // the OLDEST matching prefetch: a caller that recycles its host buffers issues the next cycle's prefetch
        // (same pointers) before this call, and that copy is still in flight
        for (int s = 0; s < 2; ++s) {
            const o3r_ctx::Prefetch& pf = ctx->prefetch[s];
            if (pf.valid && pf.n == n && pf.disp_type == disp_type && pf.sig == sig &&
                (!prefetched || pf.seq < ctx->prefetch[set].seq)) {
                prefetched = true; set = s;
            }
        }
        if (!prefetched && ctx->deferred.pending && (int)ctx->deferred.frames.size() == n &&
            ctx->deferred.disp_type == disp_type) {   // recorded but not issued yet (nothing ran in between): issue it now
            std::vector<const void*> dsig;
            frames_signature(ctx->deferred.frames.data(), n, dsig);
            if (dsig == sig) {
                int rcf = flush_deferred_prefetch(ctx);
                if (rcf) return rcf;
                for (int s = 0; s < 2; ++s)
                    if (ctx->prefetch[s].valid && ctx->prefetch[s].seq == ctx->prefetch_seq) { prefetched = true; set = s; }
            }
        }
        if (prefetched) ctx->prefetch[set].valid = false;
        if (!prefetched) set = ctx->free_stage_set();
        ctx->busy_set = set;
    }
    if (blur) CU(ctx->d_blur.ensure((size_t)n * p.rows * blur_step));
    std::vector<FrameDev> fd(n);
    std::vector<BlurJob> jobs(blur ? n : 0);
    bool vec = (J == 1) && (ctx->nx % 4 == 0) && (P.x0 % 4 == 0) && !label_mode;
    std::vector<FrameDev> fd_stage;   // where the H2D copies land (fd[i].disp is redirected to the blurred plane below)
    if (host_inputs) {
        int rc = stage_layout(ctx, frames, n, label_mode, J, G, set, fd);
        if (rc) return rc;
        if (!prefetched) fd_stage = fd;
    }
    for (int i = 0; i < n; ++i) {
        const o3r_frame& f = frames[i];
        FrameDev& d = fd[i];
        if (!host_inputs) {
            const int nk = (J != 1 && f.kp_xy && f.n_kp > 0) ? f.n_kp : 0;
            d.disp = (const uint8_t*)f.disp; d.disp_step = f.disp_step;
            d.bgr = f.bgr; d.bgr_step = f.bgr_step;
            d.labels = label_mode ? f.labels : nullptr; d.labels_step = f.labels_step;
            d.plane_coef = label_mode ? f.plane_coef : nullptr;
            d.kp_xy = nk ? f.kp_xy : nullptr;
            d.n_planes = label_mode ? std::max(f.n_planes, 0) : 0;
            d.n_kp = nk;
        }
        for (int k = 0; k < 12; ++k) d.T[k] = f.T[k];
        if (blur) {
            jobs[i].src = d.disp; jobs[i].sstep = d.disp_step;
            jobs[i].dst = ctx->d_blur.as<uint8_t>() + (size_t)i * p.rows * blur_step; jobs[i].dstep = blur_step;
            d.disp = jobs[i].dst; d.disp_step = blur_step;
        }
        if (!label_mode) vec = vec && ((uintptr_t)d.disp % 16 == 0) && (d.disp_step % (4 * es) == 0);
        vec = vec && ((uintptr_t)d.bgr % 4 == 0) && (d.bgr_step % 4 == 0);
    }
    P.vec = vec;
    CU(ctx->d_frames.ensure((size_t)n * sizeof(FrameDev)));
    { int rcu = upload_small(ctx, ctx->d_frames.p, fd.data(), (size_t)n * sizeof(FrameDev)); if (rcu) return rcu; }
    if (blur) {
        CU(ctx->d_blurjobs.ensure((size_t)n * sizeof(BlurJob)));
        { int rcu = upload_small(ctx, ctx->d_blurjobs.p, jobs.data(), (size_t)n * sizeof(BlurJob)); if (rcu) return rcu; }
    }

    // ---- buffers: batch-wide outputs, chunk-sized scratch
    // host inputs: chunks let the copies overlap the kernels; device inputs: one launch sequence for the whole batch
    const int chunk = std::max(1, std::min(n, (host_inputs && !prefetched) ? ctx->chunk_frames : ctx->chunk_frames_dev));
    if (prefetched && trace) {
        const bool done = cudaEventQuery(ctx->prefetch[set].ev) == cudaSuccess;
        cudaGetLastError();
        fprintf(stderr, "[o3r trace] prefetched inputs %s at entry\n", done ? "ready" : "still in flight");
    }
    if (prefetched) CU(cudaStreamWaitEvent(ctx->st, ctx->prefetch[set].ev, 0));
    const size_t per_frame_cap = (size_t)P.npix + (size_t)max_kp;
    const size_t cap_batch = per_frame_cap * n, cap_chunk = per_frame_cap * chunk;
    if (cap_batch >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "batch exceeds 2^32 samples; use fewer frames");
    const size_t n_tiles = (size_t)P.tiles_per_frame * chunk;
    uint32_t* cnt = ctx->counters.as<uint32_t>();
    // The fused bucket engine (bucket.cuh) serves the merged path of O3R_MERGE_ACCUMULATE_FUSED; everything that needs the
    // per-frame clouds themselves (single-frame calls, masks, StatisticalOutlierRemoval) or that it cannot bound runs
    // through the sort engine, as does a batch on which the device raised one of its overflow flags (second attempt).
    // Engines of the merged path, best first: the tile engine (tile.cuh: one kernel from the planes to the partial cells; dense
    // scans of a rectified-stereo Q), the bucket engine (bucket.cuh: strided scans, keypoints), the sort engine (everything).
    BkPlan bkp;
    TvPlan tvp;
    const bool fused_ok = ctx->fused() && P.want_keys && opt.merge && !opt.mask_only && !(p.sor_mean_k > 0 && J > 0);
    auto bucket_ok = [&] { return fused_ok && !ctx->bucket_off && bk_plan(ctx, frames, n, chunk, disp_type, label_mode, bkp); };
    Engine engine = fused_ok && tv_begin(ctx, P, frames, n, tvp) ? Engine::TILE : bucket_ok() ? Engine::BUCKET : Engine::SORT;
    if (trace && ctx->fused()) trace_fused_engine(ctx, engine, P, opt);
    bool inputs_resident = false;   // second attempt: the staging buffers already hold every frame
    double tr1 = 0, tr2 = 0;
    for (;;) {
        CU(ctx->tile_cnt.ensure(n_tiles * 4));
        CU(ctx->tile_off.ensure(n_tiles * 4));
        CU(ctx->bbox.ensure((size_t)chunk * 6 * 4));
        CU(ctx->frame_off.ensure((size_t)(chunk + 1) * 4));
        CU(ctx->grids.ensure((size_t)chunk * sizeof(GridParams)));
        SortU32 sb{nullptr, nullptr, nullptr, nullptr};
        if (!opt.mask_only) {
            CU(ctx->vox_off.ensure((size_t)(n + 1) * 4));
            if (engine != Engine::SORT) {
                const int rc = engine == Engine::TILE ? tv_prepare(ctx, tvp, n, chunk, cap_batch)
                                                      : bk_prepare(ctx, bkp, n, cap_batch, cap_chunk);
                if (rc) return rc;
            } else if (P.want_keys) {
                CU(ctx->pts.ensure(cap_chunk * 16));
                CU(ctx->vox.ensure(cap_batch * 16));
                int rc = carve_sort_u32(ctx, cap_chunk, sb);
                if (rc) return rc;
                if (!ctx->retain()) FILL(cnt + CNT_CELLBB, 24, FILL_CELLBB);
                // (a chunk that could hold 2^30 per-frame voxels goes around it: k_cell_prereduce's look-back word counts 30 bits)
                ctx->tiled_now = ctx->tiled() && !(ctx->tiled_poor && (ctx->tiled_batches % 16) != 0) && cap_chunk < kRsWideSeg;
                ++ctx->tiled_batches;
                if (ctx->tiled_now) {   // worst case one partial per item; never reached in practice (~1/8)
                    CU(ctx->partials.ensure(cap_batch * sizeof(o3r_cell)));
                    CU(ctx->pr_status.ensure(((size_t)cdiv(cap_chunk, kPrTile) + 16) * 4));
                    ZERO(cnt + CNT_PART, 8);
                }
            } else {
                CU(ctx->pts.ensure(cap_batch * 16));
            }
            ZERO(cnt + CNT_BASE, 4);
            ZERO(ctx->vox_off.p, 4);
        }
        if (!opt.mask_only) ctx->last_is_vox = P.want_keys;
        uint32_t* goff = ctx->vox_off.as<uint32_t>();

        for (int f0 = 0; f0 < n; f0 += chunk) {
            const int nc = std::min(chunk, n - f0);
            if (host_inputs && !prefetched && !inputs_resident) {  // H2D of this chunk on the copy stream; the compute stream waits for its event only
                int rc = stage_copy(ctx, frames, fd_stage, f0, nc, label_mode, G);
                if (rc) return rc;
                cudaEvent_t ev = ctx->chunk_event(f0 / chunk);
                CU(cudaEventRecord(ev, ctx->st_copy));
                CU(cudaStreamWaitEvent(ctx->st, ev, 0));
            }
            const FrameDev* fr = ctx->d_frames.as<FrameDev>() + f0;
            if (blur) {
                const int rx0 = P.x0, rx1 = p.cols - p.bounding_box, ry0 = p.bounding_box, ry1 = p.rows - p.bounding_box;
                if (rx1 > rx0 && ry1 > ry0) {
                    const dim3 g(cdiv(rx1 - rx0, kBlurStrip), cdiv(ry1 - ry0, blur_rows(p.blur_mode)), nc);
                    const size_t sm = blur_smem(p.blur_kernel, p.blur_mode);
                    const BlurJob* bj = ctx->d_blurjobs.as<BlurJob>() + f0;
                    if (p.blur_mode == O3R_BLUR_BILATERAL) {
                        BilateralLut L;
                        int rcl = bilateral_lut(ctx, p.blur_kernel, &L);
                        if (rcl) return rcl;
                        const dim3 gb(cdiv(rx1 - rx0, kBilW), cdiv(ry1 - ry0, kBilTY), nc);
                        LAUNCH(k_bilateral, gb, dim3(kBilTX, kBilTY), bilateral_smem(L.radius, L.maxk), bj, L, p.rows, p.cols, rx0, ry0, rx1, ry1);
                    } else if (p.blur_mode == O3R_BLUR_MEDIAN)
                        LAUNCH_N("k_blur_median", (k_blur<O3R_BLUR_MEDIAN>), g, kBlurRows, sm, bj, p.rows, p.cols, p.blur_kernel, rx0, ry0, rx1, ry1);
                    else
                        LAUNCH_N("k_blur_box", (k_blur<O3R_BLUR_BOX>), g, kBlurRows, sm, bj, p.rows, p.cols, p.blur_kernel, rx0, ry0, rx1, ry1);
                }
            }
            // tile engine: planes -> partial cells of the chunk, per-frame voxel counts, exact bboxes; bucket engine: the same through
            // hist -> scan -> scatter -> reduce; sort engine: stage A, whose V1 mode writes the chunk scratch and whose
            // dont_downsample mode writes the batch buffer at the running base
            float4* pts_out = ctx->pts.as<float4>();
            const uint32_t* base_a = P.want_keys ? nullptr : cnt + CNT_BASE;
            uint32_t* goff_a = P.want_keys ? nullptr : goff + f0;
            int rc = with_disp_type(disp_type, [&](auto dt) {
                constexpr int DT = decltype(dt)::value;
                if (engine == Engine::TILE) return tv_run_chunk<DT>(ctx, P, tvp, f0, nc, n);
                if (engine == Engine::BUCKET) return bk_run_chunk<DT>(ctx, P, bkp, f0 / chunk, f0, nc, n, cap_chunk);
                return launch_stage_a<DT>(ctx, P, fr, nc, opt, pts_out, sb.k0, base_a, goff_a);
            });
            if (rc) return rc;
            if (engine != Engine::SORT) continue;
            if (opt.mask_only) { ctx->busy_set = -1; return O3R_OK; }   // (single frame; the last batch's state is untouched)
            const float4* vg_pts = ctx->pts.as<float4>();
            const uint32_t* vg_off = ctx->frame_off.as<uint32_t>();
            if (P.want_keys && p.sor_mean_k > 0 && J > 0) {
                // StatisticalOutlierRemoval first (pose_functions.cpp:1673-1686); the VoxelGrid then sees the filtered cloud, so
                // its bbox, grid and leaf indices are recomputed from the kept points
                rc = sor_filter(ctx, sb, vg_pts, vg_off, nc, per_frame_cap, p.sor_mean_k, p.sor_stddev_mul);
                if (rc) return rc;
                vg_pts = ctx->sor_pts.as<float4>();
                vg_off = ctx->sor_off.as<uint32_t>();
                const uint32_t tl = std::max(1u, cdiv(per_frame_cap, kTileV));
                FILL(ctx->bbox.as<uint32_t>(), (size_t)(nc) * 24, FILL_BBOX);
                LAUNCH(k_bbox_pts, dim3(tl, nc), kThreads, 0, vg_pts, vg_off, 0, ctx->bbox.as<uint32_t>());
                LAUNCH(k_grid_params, cdiv(nc, 64), 64, 0, nc, ctx->bbox.as<uint32_t>(), ctx->inv_f, ctx->inv_f, ctx->inv_f,
                       ctx->grids.as<GridParams>());
                LAUNCH(k_vg_key, dim3(std::min<uint32_t>(std::max(1u, cdiv(per_frame_cap, kThreads)), 148 * 4), nc), kThreads, 0, vg_pts,
                       vg_off, ctx->grids.as<GridParams>(), 0, sb.k0);
            }
            if (P.want_keys) {  // per-frame VoxelGrid, leaf voxel_size / 5 (pose_functions.cpp:1698), appended at the base
                rc = vg_sorted_reduce(ctx, sb, vg_pts, vg_off, nc, per_frame_cap,
                                      ctx->grids.as<GridParams>(), ctx->inv_f, ctx->inv_f, ctx->inv_f, 0, 0,
                                      ctx->vox.as<float4>(), goff + f0, nullptr, nullptr, !ctx->retain(), cnt + CNT_BASE);
                if (rc) return rc;
                if (ctx->tiled_now) {   // group the chunk's voxel centroids by combined-grid cell, tile by tile
                    const uint32_t pt = cdiv(cap_chunk, kPrTile);
                    uint32_t* stw = ctx->pr_status.as<uint32_t>();
                    ZERO(stw, ((size_t)pt + 16) * 4);
                    ZERO(cnt + CNT_PARTCHUNK, 4);
                    LAUNCH(k_cell_prereduce, pt, kThreads, 0, ctx->vox.as<float4>(), cnt + CNT_BASE, cnt + CNT_VOX, ctx->inv_c,
                           ctx->inv_cz, ctx->partials.as<o3r_cell>(), cnt + CNT_PART, cnt + CNT_PARTCHUNK, stw, stw + pt);
                    LAUNCH(k_add_u32, 1, 32, 0, cnt + CNT_PART, cnt + CNT_PARTCHUNK);
                }
                LAUNCH(k_add_base, 1, 32, 0, cnt + CNT_BASE, cnt + CNT_VOX, goff + f0 + nc);
            } else {
                LAUNCH(k_add_base, 1, 32, 0, cnt + CNT_BASE, cnt + CNT_PTS, goff + f0 + nc);
            }
        }

        // ---- per-frame output offsets (+ the combined-grid cell range) back to the host: the one sync of the frame path
        const size_t offs_words = (size_t)n + 3 + ((size_t)n + 3) / 4 + 1;   // offsets / counts, two flag words, n flag bytes
        if (ctx->h_offs_cap < offs_words) {
            if (ctx->h_offs) cudaFreeHost(ctx->h_offs);
            ctx->h_offs_cap = std::max<size_t>(offs_words, 256);
            CU(cudaMallocHost((void**)&ctx->h_offs, ctx->h_offs_cap * 4));
        }
        if (engine != Engine::SORT) {   // per-frame counts and the engine's flags
            const int rc = engine == Engine::TILE ? tv_read_back(ctx, n) : bk_read_back(ctx, n);
            if (rc) return rc;
        } else {
            CU(cudaMemcpyAsync(ctx->h_offs, goff, (size_t)(n + 1) * 4, cudaMemcpyDeviceToHost, ctx->st));
        }
        ctx->last_has_cellbb = ctx->last_is_vox && !ctx->retain();
        if (ctx->last_has_cellbb)
            CU(cudaMemcpyAsync(ctx->h_counters + CNT_CELLBB, cnt + CNT_CELLBB, 24, cudaMemcpyDeviceToHost, ctx->st));
        // the kernels of this call are queued: now issue the copies of a recorded prefetch (next cycle's inputs).  The
        // staging set they go to is not the one these kernels read.
        if (ctx->deferred.pending && !opt.mask_only) {
            int rcf = flush_deferred_prefetch(ctx);
            if (rcf) return rcf;
        }
        ctx->last_has_partials = ctx->last_is_vox && ((ctx->tiled() && ctx->tiled_now) || engine != Engine::SORT);
        if (ctx->last_has_partials)
            CU(cudaMemcpyAsync(ctx->h_counters + CNT_PART, cnt + CNT_PART, 4, cudaMemcpyDeviceToHost, ctx->st));
        tr1 = now_ms();
        CU(cudaStreamSynchronize(ctx->st));
        tr2 = now_ms();
        if (engine != Engine::SORT) {
            const Verdict v = engine == Engine::TILE ? tv_verdict(ctx, tvp, n) : bk_verdict(ctx, n);
            if (v != Verdict::ACCEPT) {   // rerun from the staging buffers, with this engine or the next one
                inputs_resident = true;
                if (v == Verdict::NEXT_ENGINE) engine = engine == Engine::TILE && bucket_ok() ? Engine::BUCKET : Engine::SORT;
                continue;
            }
            ctx->h_offs[0] = 0;   // per-frame counts -> offsets
            for (int i = 0; i < n; ++i) ctx->h_offs[i + 1] += ctx->h_offs[i];
        }
        break;
    }
    ctx->last_engine = engine;
    ctx->busy_set = -1;
    ctx->last_partials = ctx->last_has_partials ? ctx->h_counters[CNT_PART] : 0;
    // The tile pre-reduction pays only when it reduces: a 40-byte partial replaces a 16-byte voxel in the merge.  On grids
    // finer than the point spacing (e.g. 4K at voxel_size 0.01) nearly every voxel is its own cell: merge the voxels then.
    if (ctx->last_has_partials && engine == Engine::SORT) {
        ctx->tiled_poor = ctx->last_partials * 2 > ctx->h_offs[n];
        if (ctx->tiled_poor) { ctx->last_has_partials = false; ctx->last_partials = 0; }
    }
    if (ctx->last_has_cellbb) memcpy(ctx->last_cellbb, ctx->h_counters + CNT_CELLBB, 24);
    ctx->last_off.assign(ctx->h_offs, ctx->h_offs + n + 1);
    ctx->last_n = n;
    ctx->last_total = ctx->last_off[n];
    if (frame_counts)
        for (int i = 0; i < n; ++i) frame_counts[i] = ctx->last_off[i + 1] - ctx->last_off[i];
    if (!opt.merge || (ctx->comm && !ctx->retain())) return O3R_OK;   // with a communicator, o3r_exchange_cycle merges the cycle
    const float4* outp = ctx->last_is_vox ? ctx->vox.as<float4>() : ctx->pts.as<float4>();
    if (ctx->retain()) {
        const size_t base = ctx->n_cloud;
        const int rca = cloud_append_dev(ctx, outp, ctx->last_total);
        if (rca) return rca;
        if (rt_shard)   // rank r's frame i is the cycle's frame i * world + r
            for (int i = 0; i < n; ++i)
                if (ctx->last_off[i + 1] > ctx->last_off[i])
                    ctx->rt_frames.push_back({base + ctx->last_off[i], rt_cycle, (uint32_t)i * (uint32_t)ctx->world + (uint32_t)ctx->rank});
        return O3R_OK;
    }
    const int* bbp = ctx->last_has_cellbb ? ctx->last_cellbb : nullptr;
    if (engine != Engine::SORT && ctx->last_partials == 0) return O3R_OK;   // nothing valid in the whole batch
    const int rcm = ctx->last_has_partials ? acc_merge_cells(ctx, ctx->partials.as<o3r_cell>(), ctx->last_partials, bbp)
                                           : acc_merge_points(ctx, outp, ctx->last_total, bbp);
    if (trace) fprintf(stderr, "[o3r trace] frames_cloud: enqueue %.3f ms, sync wait %.3f ms, merge enqueue %.3f ms\n", tr1 - tr0, tr2 - tr1, now_ms() - tr2);
    return rcm;
}

int copy_out(o3r_ctx* ctx, const float4* src, size_t n, o3r_point* out, size_t cap, size_t* n_out) {
    if (n_out) *n_out = n;
    if (!out && cap == 0) return O3R_OK;
    if (cap < n) return ctx->fail(O3R_ERR_CAPACITY, "output buffer too small");
    if (n) {
        CU(cudaMemcpyAsync(out, src, n * 16, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
    }
    return O3R_OK;
}

}  // namespace
