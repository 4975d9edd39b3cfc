// host_register.cuh — o3r_cloud_register[_dev]: point-to-plane registration of a cloud against the resident map.  Checks
// everything first, stages host points in a buffer of its own, then queues the pivot, and every Gauss-Newton iteration as two
// launches (k_reg_step, k_reg_solve) without waiting for the GPU; one read-back of the state at the end.  It reads the resident
// map and writes only its own buffers (Registration), so the map, the change set and the last batch stay as they were.
// Kernels: register.cuh.
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "register.cuh"
#include "host_merge.cuh"

namespace {

o3r_register_params reg_defaults(const o3r_ctx* ctx) {
    o3r_register_params d;
    d.max_iterations = 20;
    d.max_distance = 3.0 * ctx->p.voxel_size;
    d.min_rotation = 1e-5;
    d.min_translation = 1e-4;
    d.degenerate_ratio = 1e-3;
    return d;
}

// T_init: finite, last row 0 0 0 1, rotation block orthonormal with det +1 (to float precision)
bool reg_rigid(const float* T) {
    for (int i = 0; i < 16; ++i)
        if (!std::isfinite(T[i])) return false;
    if (T[12] != 0.f || T[13] != 0.f || T[14] != 0.f || T[15] != 1.f) return false;
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) {
            double d = 0.0;
            for (int k = 0; k < 3; ++k) d += (double)T[k * 4 + a] * (double)T[k * 4 + b];
            if (std::fabs(d - (a == b ? 1.0 : 0.0)) > 1e-4) return false;
        }
    const double det = (double)T[0] * ((double)T[5] * T[10] - (double)T[6] * T[9]) -
                       (double)T[1] * ((double)T[4] * T[10] - (double)T[6] * T[8]) +
                       (double)T[2] * ((double)T[4] * T[9] - (double)T[5] * T[8]);
    return det > 0.0;
}

int register_impl(o3r_ctx* ctx, const o3r_point* pts, bool host_pts, size_t n, const float* T_init,
                  const o3r_register_params* prm, float* T_out, o3r_register_stats* stats) {
    if (ctx->retain())
        return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_register needs an accumulate merge mode (not O3R_MERGE_RETAIN or dont_downsample)");
    if (ctx->comm)
        return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_register with a communicator: source points would have to meet cells on other ranks");
    const o3r_register_params P = prm ? *prm : reg_defaults(ctx);
    if (P.max_iterations < 1 || !(P.max_distance > 0) || !std::isfinite(P.max_distance) || !(P.min_rotation >= 0) ||
        !std::isfinite(P.min_rotation) || !(P.min_translation >= 0) || !std::isfinite(P.min_translation) ||
        !(P.degenerate_ratio >= 0) || !(P.degenerate_ratio <= 1))
        return ctx->fail(O3R_ERR_INVALID, "o3r_register_params out of range");
    if (!reg_rigid(T_init)) return ctx->fail(O3R_ERR_INVALID, "T_init is not a rigid transform (row-major, last row 0 0 0 1)");
    if (n >= (1ull << 32)) return ctx->fail(O3R_ERR_INVALID, "too many source points for one registration (2^32 or more)");
    if (host_pts)
        for (size_t i = 0; i < n; ++i)
            if (!std::isfinite(pts[i].x) || !std::isfinite(pts[i].y) || !std::isfinite(pts[i].z))
                return ctx->fail(O3R_ERR_INVALID, "source point " + std::to_string(i) + " is not finite");
    RegState h{};
    for (int i = 0; i < 12; ++i) h.T[i] = h.T0[i] = (double)T_init[i];
    if (n) {
        Registration& G = ctx->reg;
        const float4* d_pts = reinterpret_cast<const float4*>(pts);
        if (host_pts) {
            CU(G.pts.ensure(n * 16));
            CU(cudaMemcpyAsync(G.pts.p, pts, n * 16, cudaMemcpyHostToDevice, ctx->st));
            d_pts = G.pts.as<float4>();
        }
        const uint32_t blocks = std::min<uint32_t>(cdiv(n, kThreads), kRegGrid);
        CU(G.part.ensure((size_t)blocks * kRegSums * 8));
        CU(G.state.ensure(sizeof(RegState)));
        if (!G.h_state) CU(cudaMallocHost((void**)&G.h_state, sizeof(RegState)));
        RegState* S = G.state.as<RegState>();
        { int rcu = upload_small(ctx, S, &h, sizeof(h)); if (rcu) return rcu; }
        RegParams rp{P.max_distance, P.min_rotation, P.min_translation, P.degenerate_ratio, ctx->inv_c, ctx->inv_cz,
                     ctx->p.min_points_per_voxel};
        double* part = G.part.as<double>();
        const ResCells R = res_cells(ctx);
        const uint32_t* n_res = ctx->counters.as<uint32_t>() + CNT_NRES;
        LAUNCH(k_reg_pivot, blocks, kThreads, 0, d_pts, n, (const RegState*)S, part);
        LAUNCH(k_reg_init, 1, 32, 0, (const double*)part, blocks, n, S);
        for (int it = 0; it < P.max_iterations; ++it) {
            LAUNCH(k_reg_step, blocks, kThreads, 0, d_pts, n, (const RegState*)S, rp, R.keys, R.acc, n_res, part);
            LAUNCH(k_reg_solve, 1, kThreads, 0, (const double*)part, blocks, rp, (uint32_t)(it == 0), S);
        }
        CU(cudaMemcpyAsync(G.h_state, S, sizeof(RegState), cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));   // (also: the caller may reuse a host `pts` now)
        h = *static_cast<const RegState*>(G.h_state);
        if (h.bad_input) return ctx->fail(O3R_ERR_INVALID, "a source point is not finite");
    }
    for (int i = 0; i < 12; ++i) T_out[i] = (float)h.T[i];
    T_out[12] = T_out[13] = T_out[14] = 0.f;
    T_out[15] = 1.f;
    if (stats) {
        stats->iterations = h.iterations;
        stats->converged = h.converged;
        stats->rank = h.rank;
        stats->n_inliers = h.n_inliers;
        stats->rms_initial = h.rms_initial;
        stats->rms_final = h.rms_final;
        for (int i = 0; i < 3; ++i) stats->pivot[i] = h.pivot[i];
        for (int i = 0; i < 36; ++i) stats->info[i] = h.info[i];
    }
    return O3R_OK;
}

}  // namespace
