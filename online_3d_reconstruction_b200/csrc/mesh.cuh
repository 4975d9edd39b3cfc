// mesh.cuh — triangulation of the resident map's height field (o3r_cloud_mesh, accumulate modes).
//
// The combined grid's leaf is (v, v, 1000) over z + 500, so the map has one centroid per (i, j) column and k: a height field
// whose mesh connects every cell to its grid neighbours.  Three passes over the sorted resident keys, each a tile of kTileV
// cells per CTA, as k_acc_emit_cnt / k_acc_emit:
//   k_mesh_vert       the vertices (o3r_cloud_downsample's records, at the offsets k_acc_emit_cnt + k_scan_u32 give them),
//                     the resident position -> vertex index map and each vertex's normal (reg_fit, register.cuh);
//   k_mesh_tri_cnt    per tile, the triangles its cells emit;
//   k_mesh_tri_emit   the triangles, at the tile's scanned offset plus the in-tile exclusive scan.
// A cell emits the quad whose A corner it is and, when (i - 1, j) is not a vertex, first the quad to its left (A missing):
// that is every quad with three or four vertices once, in ascending key of its A corner.  No atomics decide the output
// order, and the arithmetic is plain float compares: the same map gives the same bits.  Host side: host_mesh.cuh.
#pragma once
#include "register.cuh"

namespace o3r {

constexpr uint32_t kMeshNone = 0xffffffffu;     // vmap entry of a resident cell that is not a vertex
constexpr uint32_t kMeshMaxVerts = 1u << 31;   // vertex counts from here on would overflow the 32-bit triangle count

// vertex records, vmap (resident position -> vertex index or kMeshNone) and normals (3 floats per vertex)
__global__ void __launch_bounds__(kThreads) k_mesh_vert(const uint32_t* __restrict__ n_res_ptr, const uint64_t* __restrict__ res_keys,
                                                        const float4* __restrict__ res_acc, const uint4* __restrict__ res_rgb,
                                                        uint32_t min_points, const uint32_t* __restrict__ off,
                                                        float4* __restrict__ verts, uint32_t* __restrict__ vmap,
                                                        float* __restrict__ normals) {
    wait_prior();
    __shared__ uint32_t s_scan[34];
    const uint32_t n_res = *n_res_ptr;
    const uint32_t t = blockIdx.x;
    uint32_t flags = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t i = t * kTileV + threadIdx.x * 4 + j;
        if (i < n_res && __float_as_uint(res_acc[i].w) >= min_points) flags |= 1u << j;
    }
    uint32_t tot;
    uint32_t o = off[t] + block_excl_scan((uint32_t)__popc(flags), s_scan, tot);
    const long long B = 1 << 20;
    for (int j = 0; j < 4; ++j) {
        const uint32_t i = t * kTileV + threadIdx.x * 4 + j;
        if (i >= n_res) break;
        if (!(flags & (1u << j))) { vmap[i] = kMeshNone; continue; }
        verts[o] = acc_centroid(res_acc[i], res_rgb[i]);
        vmap[i] = o;
        const uint64_t key = res_keys[i];
        const int ci = (int)((long long)(key & 0x1fffffull) - B), cj = (int)((long long)((key >> 21) & 0x1fffffull) - B);
        const int ck = (int)((long long)(key >> 42) - B);
        double x0, y0, z0, nx, ny, nz;
        float3 nv = make_float3(0.f, 0.f, 0.f);
        if (reg_fit(res_keys, res_acc, n_res, min_points, ci, cj, ck, x0, y0, z0, nx, ny, nz))
            nv = make_float3((float)nx, (float)ny, (float)nz);
        normals[(size_t)o * 3 + 0] = nv.x;
        normals[(size_t)o * 3 + 1] = nv.y;
        normals[(size_t)o * 3 + 2] = nv.z;
        ++o;
    }
}

// The vertices around resident cell p: its own (a) and those of (i - 1, j), (i + 1, j), (i - 1, j + 1), (i, j + 1),
// (i + 1, j + 1), each kMeshNone when that cell is not a vertex or lies outside +-(2^20 - 1).
struct MeshNb { uint32_t a, l, r, ul, u, ur; };

__device__ __forceinline__ MeshNb mesh_nb(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vmap, uint32_t n_res,
                                          uint32_t p) {
    MeshNb nb{vmap[p], kMeshNone, kMeshNone, kMeshNone, kMeshNone, kMeshNone};
    if (nb.a == kMeshNone) return nb;
    const int lim = (1 << 20) - 1;
    const long long B = 1 << 20;
    const uint64_t key = keys[p];
    const int ci = (int)((long long)(key & 0x1fffffull) - B), cj = (int)((long long)((key >> 21) & 0x1fffffull) - B);
    const int ck = (int)((long long)(key >> 42) - B);
    // row j: sorted neighbours of p, confirmed against the key of (i -+ 1, j, k)
    if (ci > -lim && p > 0 && keys[p - 1] == reg_key(ci - 1, cj, ck)) nb.l = vmap[p - 1];
    if (ci < lim && p + 1 < n_res && keys[p + 1] == reg_key(ci + 1, cj, ck)) nb.r = vmap[p + 1];
    // row j + 1: one lower bound covers i - 1 .. i + 1 (consecutive keys)
    if (cj < lim) {
        const int i0 = ci > -lim ? ci - 1 : ci;
        uint32_t at = reg_lower_bound(keys, n_res, reg_key(i0, cj + 1, ck));
        for (int di = i0 - ci; di <= (ci < lim ? 1 : 0); ++di) {
            if (at < n_res && keys[at] == reg_key(ci + di, cj + 1, ck)) {
                const uint32_t v = vmap[at++];
                if (di < 0) nb.ul = v; else if (di == 0) nb.u = v; else nb.ur = v;
            }
        }
    }
    return nb;
}

// triangle (x, y, z) passes the gate when max |dz| over its pairs (float32), as a double, is <= max_step
__device__ __forceinline__ bool mesh_gate(float za, float zb, float zc, double max_step) {
    const float m = fmaxf(fmaxf(fabsf(__fsub_rn(za, zb)), fabsf(__fsub_rn(zb, zc))), fabsf(__fsub_rn(za, zc)));
    return (double)m <= max_step;
}

// One quad's triangles (corners A, B, C, D = (i, j), (i + 1, j), (i, j + 1), (i + 1, j + 1); kMeshNone = absent) in the
// contract's order, counter-clockwise in (i, j).  Writes them to out (when not null) and returns how many passed the gate.
__device__ __forceinline__ uint32_t mesh_quad(const float4* __restrict__ verts, uint32_t A, uint32_t Bv, uint32_t Cv, uint32_t D,
                                              double max_step, uint32_t* __restrict__ out) {
    const int present = (A != kMeshNone) + (Bv != kMeshNone) + (Cv != kMeshNone) + (D != kMeshNone);
    if (present < 3) return 0;
    uint32_t tri[6];
    int nt;
    if (present == 4) {
        const float zA = verts[A].z, zB = verts[Bv].z, zC = verts[Cv].z, zD = verts[D].z;
        if (fabsf(__fsub_rn(zA, zD)) <= fabsf(__fsub_rn(zB, zC))) {
            tri[0] = A; tri[1] = Bv; tri[2] = D; tri[3] = A; tri[4] = D; tri[5] = Cv;
        } else {
            tri[0] = A; tri[1] = Bv; tri[2] = Cv; tri[3] = Bv; tri[4] = D; tri[5] = Cv;
        }
        nt = 2;
    } else {
        if (A == kMeshNone) { tri[0] = Bv; tri[1] = D; tri[2] = Cv; }
        else if (Bv == kMeshNone) { tri[0] = A; tri[1] = D; tri[2] = Cv; }
        else if (Cv == kMeshNone) { tri[0] = A; tri[1] = Bv; tri[2] = D; }
        else { tri[0] = A; tri[1] = Bv; tri[2] = Cv; }
        nt = 1;
    }
    uint32_t m = 0;
    for (int q = 0; q < nt; ++q) {
        const uint32_t* T = tri + 3 * q;
        if (!mesh_gate(verts[T[0]].z, verts[T[1]].z, verts[T[2]].z, max_step)) continue;
        if (out) { out[3 * m + 0] = T[0]; out[3 * m + 1] = T[1]; out[3 * m + 2] = T[2]; }
        ++m;
    }
    return m;
}

// a cell's triangles: the quad to its left when (i - 1, j) is not a vertex, then its own quad
__device__ __forceinline__ uint32_t mesh_cell(const float4* __restrict__ verts, const MeshNb& nb, double max_step,
                                              uint32_t* __restrict__ out) {
    if (nb.a == kMeshNone) return 0;
    uint32_t m = 0;
    if (nb.l == kMeshNone) m = mesh_quad(verts, kMeshNone, nb.a, nb.ul, nb.u, max_step, out);
    return m + mesh_quad(verts, nb.a, nb.r, nb.u, nb.ur, max_step, out ? out + 3 * m : nullptr);
}

// per tile: the triangles its cells emit (none at all when the vertex count reached kMeshMaxVerts: the call fails)
__global__ void __launch_bounds__(kThreads) k_mesh_tri_cnt(const uint32_t* __restrict__ n_res_ptr, const uint64_t* __restrict__ keys,
                                                           const uint32_t* __restrict__ vmap, const float4* __restrict__ verts,
                                                           const uint32_t* __restrict__ n_verts, double max_step,
                                                           uint32_t* __restrict__ cnt) {
    wait_prior();
    const uint32_t n_res = *n_res_ptr;
    const uint32_t t = blockIdx.x;
    uint32_t c = 0;
    if (*n_verts < kMeshMaxVerts)
        for (int j = 0; j < 4; ++j) {
            const uint32_t p = t * kTileV + threadIdx.x * 4 + j;
            if (p >= n_res) break;
            c += mesh_cell(verts, mesh_nb(keys, vmap, n_res, p), max_step, nullptr);
        }
    c = __reduce_add_sync(kFull, c);
    __shared__ uint32_t s_c;
    if (threadIdx.x == 0) s_c = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_c, c);
    __syncthreads();
    if (threadIdx.x == 0) cnt[t] = s_c;
}

// the triangles (3 vertex indices each), tile t's at off[t] plus the in-tile exclusive scan, cells in resident order
__global__ void __launch_bounds__(kThreads) k_mesh_tri_emit(const uint32_t* __restrict__ n_res_ptr, const uint64_t* __restrict__ keys,
                                                            const uint32_t* __restrict__ vmap, const float4* __restrict__ verts,
                                                            const uint32_t* __restrict__ n_verts, double max_step,
                                                            const uint32_t* __restrict__ off, uint32_t* __restrict__ tris) {
    wait_prior();
    __shared__ uint32_t s_scan[34];
    if (*n_verts >= kMeshMaxVerts) return;
    const uint32_t n_res = *n_res_ptr;
    const uint32_t t = blockIdx.x;
    MeshNb nb[4];
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t p = t * kTileV + threadIdx.x * 4 + j;
        nb[j] = p < n_res ? mesh_nb(keys, vmap, n_res, p) : MeshNb{kMeshNone, kMeshNone, kMeshNone, kMeshNone, kMeshNone, kMeshNone};
        c += mesh_cell(verts, nb[j], max_step, nullptr);
    }
    uint32_t tot;
    size_t o = (size_t)off[t] + block_excl_scan(c, s_scan, tot);
#pragma unroll
    for (int j = 0; j < 4; ++j) o += mesh_cell(verts, nb[j], max_step, tris + 3 * o);
}

}  // namespace o3r
