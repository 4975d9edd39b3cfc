// host_mesh.cuh — o3r_cloud_mesh[_dev]: the resident map's height field as a triangle mesh.  Checks everything first, then
// queues the vertex pass (k_acc_emit_cnt, k_scan_u32, k_mesh_vert) and the triangle pass (k_mesh_tri_cnt, k_scan_u32,
// k_mesh_tri_emit), sized by the host's upper bound of the resident count, and the read-back of both totals (with the host
// copies, when there are any) behind them: one synchronise per call.  It reads the resident map and writes only its own
// buffers (Meshing), so the map, the change set, the last batch and the prefetch state stay as they were.
// Kernels: mesh.cuh.
// (host side of libo3r.so; included by o3r_api.cu, one translation unit)
#pragma once

#include "mesh.cuh"
#include "host_merge.cuh"

namespace {

// The host outputs of o3r_cloud_mesh; null for o3r_cloud_mesh_dev.
struct MeshOut { o3r_point* verts; float* normals; size_t vcap; uint32_t* tris; size_t tcap; };

int mesh_impl(o3r_ctx* ctx, double max_step, const MeshOut* out, size_t* n_verts, size_t* n_tris) {
    *n_verts = *n_tris = 0;
    if (ctx->retain())
        return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_mesh needs an accumulate merge mode (not O3R_MERGE_RETAIN or dont_downsample)");
    if (ctx->comm)
        return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_mesh with a communicator: a cell's neighbours may live on other ranks");
    if (!(max_step >= 0)) return ctx->fail(O3R_ERR_INVALID, "max_step must be >= 0 (INFINITY: no gate)");
    { int rc = refresh_nres(ctx, false); if (rc) return rc; }
    const size_t n_ub = ctx->res.n_ub;
    if (n_ub == 0) return O3R_OK;
    Meshing& M = ctx->mesh;
    const uint32_t tiles = cdiv(n_ub, kTileV);
    CU(M.vcnt.ensure((size_t)tiles * 4));
    CU(M.voff.ensure((size_t)tiles * 4));
    CU(M.tcnt.ensure((size_t)tiles * 4));
    CU(M.toff.ensure((size_t)tiles * 4));
    CU(M.tot.ensure(8));
    CU(M.vmap.ensure(n_ub * 4));
    CU(M.verts.ensure(n_ub * 16));
    CU(M.normals.ensure(n_ub * 12));
    CU(M.tris.ensure(n_ub * 2 * 12));   // a quad of 4 vertices gives 2 triangles, of 3 one: at most 2 per vertex
    if (!M.h_tot) CU(cudaMallocHost((void**)&M.h_tot, 8));
    const ResCells R = res_cells(ctx);
    const uint32_t* n_res = ctx->counters.as<uint32_t>() + CNT_NRES;
    const uint32_t min_points = ctx->p.min_points_per_voxel;
    uint32_t* tot = M.tot.as<uint32_t>();
    const float4* verts = M.verts.as<float4>();
    const uint32_t* vmap = M.vmap.as<uint32_t>();
    LAUNCH(k_acc_emit_cnt, tiles, kThreads, 0, n_res, R.acc, min_points, M.vcnt.as<uint32_t>());
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, (const uint32_t*)M.vcnt.as<uint32_t>(), M.voff.as<uint32_t>(), tiles, tot);
    LAUNCH(k_mesh_vert, tiles, kThreads, 0, n_res, R.keys, R.acc, R.rgb, min_points, (const uint32_t*)M.voff.as<uint32_t>(),
           M.verts.as<float4>(), M.vmap.as<uint32_t>(), M.normals.as<float>());
    LAUNCH(k_mesh_tri_cnt, tiles, kThreads, 0, n_res, R.keys, vmap, verts, (const uint32_t*)tot, max_step, M.tcnt.as<uint32_t>());
    LAUNCH(k_scan_u32, 1, kScanThreads, 0, (const uint32_t*)M.tcnt.as<uint32_t>(), M.toff.as<uint32_t>(), tiles, tot + 1);
    LAUNCH(k_mesh_tri_emit, tiles, kThreads, 0, n_res, R.keys, vmap, verts, (const uint32_t*)tot, max_step,
           (const uint32_t*)M.toff.as<uint32_t>(), M.tris.as<uint32_t>());
    // host outputs: up to min(cap, bound) records are copied behind the kernels; the totals decide what the call reports
    if (out) {
        const size_t nv = std::min(out->vcap, n_ub), nt = std::min(out->tcap, n_ub * 2);
        if (out->verts && nv) CU(cudaMemcpyAsync(out->verts, M.verts.p, nv * 16, cudaMemcpyDeviceToHost, ctx->st));
        if (out->normals && nv) CU(cudaMemcpyAsync(out->normals, M.normals.p, nv * 12, cudaMemcpyDeviceToHost, ctx->st));
        if (out->tris && nt) CU(cudaMemcpyAsync(out->tris, M.tris.p, nt * 12, cudaMemcpyDeviceToHost, ctx->st));
    }
    CU(cudaMemcpyAsync(M.h_tot, M.tot.p, 8, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    if (M.h_tot[0] >= kMeshMaxVerts)
        return ctx->fail(O3R_ERR_UNSUPPORTED, "o3r_cloud_mesh: the map has 2^31 or more vertices (32-bit triangle indices)");
    *n_verts = M.h_tot[0];
    *n_tris = M.h_tot[1];
    if (!out) return O3R_OK;
    if (!out->verts && !out->normals && !out->tris && out->vcap == 0 && out->tcap == 0) return O3R_OK;   // size query
    if (out->vcap < *n_verts || out->tcap < *n_tris) return ctx->fail(O3R_ERR_CAPACITY, "output buffer too small");
    return O3R_OK;
}

}  // namespace
