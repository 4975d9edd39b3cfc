// stage_a.cuh — fused per-frame kernel: validity mask + Q reprojection + rigid transform + colour +
// VoxelGrid leaf index + stable stream compaction with coalesced float4 stores.
//
// Replaces createSingleImgPtCloud (pose_functions.cpp:1030-1134) + transformPtCloud (:1358-1362) and the
// first pass of pcl::VoxelGrid::applyFilter (leaf index) for a whole batch of frames per launch.
//
// Work decomposition: a frame's output order is "keypoints (ORB order), then the row-major grid scan"
// (pose_functions.cpp:1057-1130), so each frame is cut into tiles of 1024 consecutive samples of that
// order; one 256-thread CTA owns one tile, 4 consecutive samples per thread (one 32-bit load of u8
// disparity, three 32-bit loads of BGR when the row geometry allows).  Two launches:
//   k_pre   counts valid samples per tile and reduces the per-frame bbox of the transformed points
//           (PCL getMinMax3D — needed before any leaf index can be formed),
//   k_emit  recomputes the samples, compacts them through shared memory at the tile's scanned offset
//           and writes points (16 B) + leaf index (4 B) with fully coalesced stores.
// Disparity is read twice (it is 6 % of the traffic and L2-resident on the second read); colour and
// outputs move exactly once.
#pragma once
#include "common.cuh"

namespace o3r {

constexpr int kTileA = 1024;

struct AParams {
    int rows, cols, x0, bb, J, nx, ny;
    uint32_t npix;            // nx * ny grid samples per frame (0 when J == 0)
    int kp_tiles;             // leading tiles that hold keypoints (J != 1)
    int tiles_per_frame;
    int label_mode;           // labels + plane coefficients instead of a disparity plane
    int canon;                // Q has the stereo-rectified sparsity (see reproject())
    int use_lut;              // u8 disparity && canon: 1/(Q32*d+Q33) from a 256-entry table
    int vec;                  // J == 1 and 4-sample groups are row-contiguous and load-aligned
    int thr_i;                // u8: valid iff d > thr_i  (== (double)d > min_disparity)
    int want_bbox, want_keys;
    double min_disp, div;
    double q[16];
    const double* lut_r;      // [256] 1.0 / (q14*d + q15)
    const float* lut_z;       // [256] (float)(q11 * lut_r[d])
    float leaf_inv[3];        // per-frame grid (voxel_size / 5)
};

// ---- disparity sample as a double (pose_functions.cpp:1098-1104, :968-971) --------------------------------
template <int DT>
__device__ __forceinline__ double disp_scalar(const AParams& P, const FrameDev& F, int x, int y) {
    if (P.label_mode) {
        const int l = F.labels[(size_t)y * F.labels_step + x];
        if (l == 0 || l > F.n_planes) return 0.0;
        const double* c = F.plane_coef + 3 * (l - 1);
        const double t0 = __dmul_rn(__dmul_rn(1.0, c[0]), (double)x);
        const double t1 = __dmul_rn(__dmul_rn(1.0, c[1]), (double)y);
        return __dadd_rn(__dadd_rn(t0, t1), __dmul_rn(1.0, c[2]));
    }
    const uint8_t* row = F.disp + (size_t)y * F.disp_step;
    if (DT == O3R_DISP_U8) return (double)row[x];
    if (DT == O3R_DISP_U16) return __ddiv_rn((double)((const uint16_t*)row)[x], P.div);
    if (DT == O3R_DISP_F32) return (double)((const float*)row)[x];
    return ((const double*)row)[x];
}

// ---- Q * [x y d 1]^T, scale by 1/w, float casts (pose_functions.cpp:1110-1117) -----------------------------
// cv::Mat_<double> 4x4 * 4x1 sums each row left to right; `/= w` multiplies by 1.0/w.  With the
// rectified-stereo sparsity (q1=q2=q4=q6=q8=q9=q10=q12=q13=0) the zero products drop out exactly:
//   v0 = q0*x + q3, v1 = q5*y + q7, v2 = q11, v3 = q14*d + q15.
// `w` receives the homogeneous coordinate v3 (its magnitude bounds the pixel footprint of a distance at that depth: tile.cuh)
__device__ __forceinline__ void reproject_w(const AParams& P, int x, int y, double d, float& X, float& Y, float& Z, double& w) {
    const double dx = (double)x, dy = (double)y;
    double v0, v1, v2, v3;
    if (P.canon) {
        v0 = __dadd_rn(__dmul_rn(P.q[0], dx), P.q[3]);
        v1 = __dadd_rn(__dmul_rn(P.q[5], dy), P.q[7]);
        v2 = P.q[11];
        v3 = __dadd_rn(__dmul_rn(P.q[14], d), P.q[15]);
    } else {
        v0 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.q[0], dx), __dmul_rn(P.q[1], dy)), __dmul_rn(P.q[2], d)), P.q[3]);
        v1 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.q[4], dx), __dmul_rn(P.q[5], dy)), __dmul_rn(P.q[6], d)), P.q[7]);
        v2 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.q[8], dx), __dmul_rn(P.q[9], dy)), __dmul_rn(P.q[10], d)), P.q[11]);
        v3 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.q[12], dx), __dmul_rn(P.q[13], dy)), __dmul_rn(P.q[14], d)), P.q[15]);
    }
    const double s = __ddiv_rn(1.0, v3);
    X = __double2float_rn(__dmul_rn(v0, s));
    Y = __double2float_rn(__dmul_rn(v1, s));
    Z = __double2float_rn(__dmul_rn(v2, s));
    w = v3;
}
__device__ __forceinline__ void reproject(const AParams& P, int x, int y, double d, float& X, float& Y, float& Z) {
    double w;
    reproject_w(P, x, y, d, X, Y, Z, w);
}

struct Samp {
    uint32_t mask;       // bit j: sample j valid
    float x[4], y[4], z[4];
    int px[4], py[4];
    int vec_row;         // 1: the four samples are (px[0]..px[0]+3, py[0]) and colour can be loaded as 3 words
};

// Evaluates the thread's 4 samples of `tile` of frame F: validity + camera-frame point.
template <int DT>
__device__ __forceinline__ void eval4(const AParams& P, const FrameDev& F, const double* rl, const float* zl,
                                      int tile, Samp& S) {
    S.mask = 0;
    S.vec_row = 0;
    const int tid = threadIdx.x;
    if (tile < P.kp_tiles) {  // keypoints first, ORB order, int truncation (pose_functions.cpp:1059-1062)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i = tile * kTileA + tid * 4 + j;
            if (i < F.n_kp) {
                const int x = (int)F.kp_xy[2 * i], y = (int)F.kp_xy[2 * i + 1];
                if (x >= P.x0 && x < P.cols - P.bb && y >= P.bb && y < P.rows - P.bb) {
                    const double d = disp_scalar<DT>(P, F, x, y);
                    if (d > P.min_disp) {
                        S.mask |= 1u << j;
                        S.px[j] = x; S.py[j] = y;
                        reproject(P, x, y, d, S.x[j], S.y[j], S.z[j]);
                    }
                }
            }
        }
        return;
    }
    const uint32_t s0 = (uint32_t)(tile - P.kp_tiles) * kTileA + tid * 4;
    if (s0 >= P.npix) return;
    if (P.vec) {  // J == 1, nx % 4 == 0: the group lies in one row and is load-aligned
        const int r = s0 / P.nx, c = s0 - r * P.nx;
        const int y = P.bb + r, xb = P.x0 + c;
        S.vec_row = 1;
        const uint8_t* row = F.disp + (size_t)y * F.disp_step;
        if (DT == O3R_DISP_U8) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(row + xb);
            if (P.use_lut) {
                const double vy = __dadd_rn(__dmul_rn(P.q[5], (double)y), P.q[7]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int d = (w >> (8 * j)) & 255;
                    S.px[j] = xb + j; S.py[j] = y;
                    if (d > P.thr_i) {
                        S.mask |= 1u << j;
                        const double s = rl[d];
                        const double v0 = __dadd_rn(__dmul_rn(P.q[0], (double)(xb + j)), P.q[3]);
                        S.x[j] = __double2float_rn(__dmul_rn(v0, s));
                        S.y[j] = __double2float_rn(__dmul_rn(vy, s));
                        S.z[j] = zl[d];
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int d = (w >> (8 * j)) & 255;
                    S.px[j] = xb + j; S.py[j] = y;
                    if (d > P.thr_i) {
                        S.mask |= 1u << j;
                        reproject(P, xb + j, y, (double)d, S.x[j], S.y[j], S.z[j]);
                    }
                }
            }
        } else {
            double dv[4];
            if (DT == O3R_DISP_U16) {
                const uint2 w = *reinterpret_cast<const uint2*>(row + 2 * (size_t)xb);
                dv[0] = __ddiv_rn((double)(w.x & 0xffffu), P.div); dv[1] = __ddiv_rn((double)(w.x >> 16), P.div);
                dv[2] = __ddiv_rn((double)(w.y & 0xffffu), P.div); dv[3] = __ddiv_rn((double)(w.y >> 16), P.div);
            } else if (DT == O3R_DISP_F32) {
                const float4 w = *reinterpret_cast<const float4*>(row + 4 * (size_t)xb);
                dv[0] = (double)w.x; dv[1] = (double)w.y; dv[2] = (double)w.z; dv[3] = (double)w.w;
            } else {
                const double2 a = *reinterpret_cast<const double2*>(row + 8 * (size_t)xb);
                const double2 b = *reinterpret_cast<const double2*>(row + 8 * (size_t)xb + 16);
                dv[0] = a.x; dv[1] = a.y; dv[2] = b.x; dv[3] = b.y;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                S.px[j] = xb + j; S.py[j] = y;
                if (dv[j] > P.min_disp) {
                    S.mask |= 1u << j;
                    reproject(P, xb + j, y, dv[j], S.x[j], S.y[j], S.z[j]);
                }
            }
        }
        return;
    }
    // generic stride / unaligned rows: one sample at a time (pose_functions.cpp:1094-1128)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t s = s0 + j;
        if (s < P.npix) {
            const int r = s / P.nx, c = s - r * P.nx;
            const int y = P.bb + r * P.J, x = P.x0 + c * P.J;
            S.px[j] = x; S.py[j] = y;
            const double d = disp_scalar<DT>(P, F, x, y);
            if (d > P.min_disp) {
                S.mask |= 1u << j;
                reproject(P, x, y, d, S.x[j], S.y[j], S.z[j]);
            }
        }
    }
}

__device__ __forceinline__ void load_lut(const AParams& P, double* rl, float* zl) {
    if (P.use_lut) {
        rl[threadIdx.x] = P.lut_r[threadIdx.x];
        zl[threadIdx.x] = P.lut_z[threadIdx.x];
    }
    __syncthreads();
}

// ---- pass 1: per-tile valid counts, per-frame bbox of the transformed points, optional mask --------------
template <int DT>
__global__ void __launch_bounds__(kThreads) k_pre(AParams P, const FrameDev* __restrict__ frames,
                                                  uint32_t* __restrict__ tile_cnt, uint32_t* __restrict__ bbox,
                                                  uint8_t* __restrict__ mask_out) {
    wait_prior();
    __shared__ double rl[256];
    __shared__ float zl[256];
    __shared__ uint32_t s_red[8];
    const int tile = blockIdx.x, f = blockIdx.y;
    const FrameDev& F = frames[f];
    if (threadIdx.x < 8) s_red[threadIdx.x] = (threadIdx.x < 3) ? 0xffffffffu : 0u;  // min x3, max x3, count
    load_lut(P, rl, zl);
    Samp S;
    eval4<DT>(P, F, rl, zl, tile, S);
    uint32_t mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u};
    if (P.want_bbox) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (S.mask & (1u << j)) {
                float tx, ty, tz;
                xform(F.T, S.x[j], S.y[j], S.z[j], tx, ty, tz);
                const uint32_t ox = f2ord(tx), oy = f2ord(ty), oz = f2ord(tz);
                mn[0] = min(mn[0], ox); mx[0] = max(mx[0], ox);
                mn[1] = min(mn[1], oy); mx[1] = max(mx[1], oy);
                mn[2] = min(mn[2], oz); mx[2] = max(mx[2], oz);
            }
    }
    if (mask_out && tile >= P.kp_tiles) {
        const uint32_t s0 = (uint32_t)(tile - P.kp_tiles) * kTileA + threadIdx.x * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (s0 + j < P.npix) mask_out[(size_t)f * P.npix + s0 + j] = (S.mask >> j) & 1u;
    }
    const uint32_t cnt = __reduce_add_sync(kFull, (uint32_t)__popc(S.mask));
    if (P.want_bbox) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            mn[a] = __reduce_min_sync(kFull, mn[a]);
            mx[a] = __reduce_max_sync(kFull, mx[a]);
        }
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_red[6], cnt);
        if (P.want_bbox && cnt) {
#pragma unroll
            for (int a = 0; a < 3; ++a) { atomicMin(&s_red[a], mn[a]); atomicMax(&s_red[3 + a], mx[a]); }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) tile_cnt[(size_t)f * P.tiles_per_frame + tile] = s_red[6];
    if (P.want_bbox && threadIdx.x < 6 && s_red[6]) {
        if (threadIdx.x < 3) atomicMin(&bbox[f * 6 + threadIdx.x], s_red[threadIdx.x]);
        else atomicMax(&bbox[f * 6 + threadIdx.x], s_red[threadIdx.x]);
    }
}

// ---- after the tile scan: frame offsets + per-frame VoxelGrid parameters ------------------------------------
// `goff` (optional): the batch-wide offsets of this chunk's frames = *out_base + chunk-local offset.
__global__ void k_a_post(int n_frames, int tiles_per_frame, const uint32_t* __restrict__ tile_off,
                         const uint32_t* __restrict__ total, const uint32_t* __restrict__ bbox, float ix, float iy,
                         float iz, int want_grid, uint32_t* __restrict__ frame_off, GridParams* __restrict__ grids,
                         const uint32_t* __restrict__ out_base, uint32_t* __restrict__ goff) {
    wait_prior();
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f > n_frames) return;
    const uint32_t o = (f == n_frames) ? *total : tile_off[(size_t)f * tiles_per_frame];
    frame_off[f] = o;
    if (goff && f < n_frames) goff[f] = *out_base + o;
    if (f < n_frames && want_grid) grids[f] = make_grid(bbox + 6 * f, ix, iy, iz);
}

// ---- pass 2: recompute, compact, emit points (+ leaf index) -------------------------------------------------
template <int DT>
__global__ void __launch_bounds__(kThreads) k_emit(AParams P, const FrameDev* __restrict__ frames,
                                                   const uint32_t* __restrict__ tile_off,
                                                   const uint32_t* __restrict__ frame_off,
                                                   const GridParams* __restrict__ grids,
                                                   float4* __restrict__ pts, uint32_t* __restrict__ keys,
                                                   const uint32_t* __restrict__ out_base) {
    wait_prior();
    __shared__ double rl[256];
    __shared__ float zl[256];
    __shared__ uint32_t s_scan[34];
    __shared__ __align__(128) float4 s_pts[kTileA];
    __shared__ uint32_t s_keys[kTileA];
    const int tile = blockIdx.x, f = blockIdx.y;
    const FrameDev& F = frames[f];
    load_lut(P, rl, zl);
    Samp S;
    eval4<DT>(P, F, rl, zl, tile, S);
    uint32_t total;
    const uint32_t off = block_excl_scan((uint32_t)__popc(S.mask), s_scan, total);
    if (total == 0) return;
    if (S.mask) {
        uint32_t rgb[4];
        if (S.vec_row) {
            const uint32_t* c = reinterpret_cast<const uint32_t*>(F.bgr + (size_t)S.py[0] * F.bgr_step + 3 * (size_t)S.px[0]);
            const uint32_t w0 = __ldcs(c), w1 = __ldcs(c + 1), w2 = __ldcs(c + 2);
            rgb[0] = w0 & 0x00ffffffu;
            rgb[1] = (w0 >> 24) | ((w1 & 0xffffu) << 8);
            rgb[2] = (w1 >> 16) | ((w2 & 0xffu) << 16);
            rgb[3] = w2 >> 8;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (S.mask & (1u << j)) {
                    const uint8_t* c = F.bgr + (size_t)S.py[j] * F.bgr_step + 3 * (size_t)S.px[j];
                    rgb[j] = ((uint32_t)c[2] << 16) | ((uint32_t)c[1] << 8) | (uint32_t)c[0];
                }
        }
        GridParams G;
        if (P.want_keys) G = grids[f];
        uint32_t o = off;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (S.mask & (1u << j)) {
                float tx, ty, tz;
                xform(F.T, S.x[j], S.y[j], S.z[j], tx, ty, tz);
                s_pts[o] = make_float4(tx, ty, tz, __uint_as_float(rgb[j]));
                if (P.want_keys) s_keys[o] = G.passthrough ? 0u : vg_rel_idx(G, tx, ty, tz);
                ++o;
            }
    }
    // The tile's points leave as ONE bulk copy (TMA, shared -> global, issued by one thread): the 16-byte records are
    // contiguous in shared memory and in the output, so no thread has to issue store instructions for them.  The writers'
    // generic-proxy stores are fenced into the async proxy before the barrier.
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    const uint32_t base = tile_off[(size_t)f * P.tiles_per_frame + tile];
    const bool pass = P.want_keys && grids[f].passthrough;
    const uint32_t fbase = frame_off[f];
    if (out_base) pts += *out_base;   // batch-wide output position of this chunk
    if (threadIdx.x == 0) {
        const uint32_t src = (uint32_t)__cvta_generic_to_shared(s_pts);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(pts + base), "r"(src), "r"(total * 16u)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    if (P.want_keys)
        for (uint32_t i = threadIdx.x; i < total; i += kThreads)
            keys[base + i] = pass ? (base + i - fbase) : s_keys[i];  // passthrough: identity order
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem is read before the CTA retires
}

}  // namespace o3r
