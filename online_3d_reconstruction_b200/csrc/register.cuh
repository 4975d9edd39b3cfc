// register.cuh — point-to-plane registration of a cloud against the resident map (o3r_cloud_register, accumulate modes).
//
// The combined grid's leaf is (v, v, 1000) over z + 500, so every map cell is a column and a point's map surface is found
// with one key lookup.  One Gauss-Newton iteration is two kernels: k_reg_step (one thread per source point, fixed grid)
// transforms the point, finds its cell and the 3 x 3 cells around it in the sorted resident keys, fits the local plane,
// gates the residual and leaves its CTA's sums of the normal equations in double; k_reg_solve (one CTA) adds the CTA
// partials in CTA order, solves the 6 x 6 system by a symmetric eigen-decomposition and composes the update into the
// device-resident transform.  No float atomics: the same inputs give the same bits.  Host side: host_register.cuh.
#pragma once
#include "voxel.cuh"

namespace o3r {

constexpr int kRegSums = 32;      // per CTA: 21 of J^T J (upper triangle, row-major), 6 of J^T r, inliers, sum r^2, pad
constexpr int kRegGrid = 148 * 4; // CTAs of k_reg_step / k_reg_pivot at most (a fixed grid: the sums' order depends on n only)
constexpr double kRegFitCond = 1e-3;   // a plane fit is singular unless det(M) > this * Suu * Sww * S1 (Hadamard bound)

// what the iterations keep on the device; read back once at the end of a call
struct RegState {
    double T[12];         // current transform, row-major 3 x 4
    double T0[12];        // T_init
    double pivot[3];
    double rms_initial, rms_final;
    double info[36];
    uint32_t iterations, converged, rank, n_inliers;
    uint32_t done, bad_input;
};

struct RegParams {
    double max_distance, min_rotation, min_translation, degenerate_ratio;
    float inv_c, inv_cz;
    uint32_t min_points;
};

// the lower bound of key k in the resident keys
__device__ __forceinline__ uint32_t reg_lower_bound(const uint64_t* __restrict__ keys, uint32_t n, uint64_t k) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (keys[mid] < k) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// 64-bit absolute key of combined-grid cell (i, j, k); fields are in range (the caller checked)
__device__ __forceinline__ uint64_t reg_key(int i, int j, int k) {
    const long long B = 1 << 20;
    return ((uint64_t)(k + B) << 42) | ((uint64_t)(j + B) << 21) | (uint64_t)(i + B);
}

// Reduces `v` over the CTA in a fixed order (warp shuffles, then warps in index order); thread 0 gets the total.
__device__ __forceinline__ double reg_block_sum(double v, double* sm) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(kFull, v, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < kWarps; ++w) s += sm[w];
    __syncthreads();
    return s;
}

__device__ __forceinline__ void reg_apply(const double* T, float x, float y, float z, double& ox, double& oy, double& oz) {
    const double px = x, py = y, pz = z;
    ox = T[0] * px + T[1] * py + T[2] * pz + T[3];
    oy = T[4] * px + T[5] * py + T[6] * pz + T[7];
    oz = T[8] * px + T[9] * py + T[10] * pz + T[11];
}

// per CTA: sums of T_init * p over its points (x, y, z) and a non-finite flag
__global__ void __launch_bounds__(kThreads) k_reg_pivot(const float4* __restrict__ pts, size_t n, const RegState* __restrict__ S,
                                                        double* __restrict__ part) {
    wait_prior();
    __shared__ double sm[kWarps];
    __shared__ double T[12];
    if (threadIdx.x < 12) T[threadIdx.x] = S->T0[threadIdx.x];
    __syncthreads();
    double sx = 0.0, sy = 0.0, sz = 0.0, bad = 0.0;
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        const float4 p = pts[i];
        if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) { bad = 1.0; continue; }
        double x, y, z;
        reg_apply(T, p.x, p.y, p.z, x, y, z);
        sx += x; sy += y; sz += z;
    }
    const double v[4] = {sx, sy, sz, bad};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const double s = reg_block_sum(v[q], sm);
        if (threadIdx.x == 0) part[(size_t)blockIdx.x * 4 + q] = s;
    }
}

// the pivot (centroid of T_init * p) from the CTA sums in CTA order; flags non-finite input
__global__ void k_reg_init(const double* __restrict__ part, uint32_t blocks, size_t n, RegState* __restrict__ S) {
    wait_prior();
    if (threadIdx.x != 0) return;
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (uint32_t b = 0; b < blocks; ++b)
        for (int q = 0; q < 4; ++q) s[q] += part[(size_t)b * 4 + q];
    for (int q = 0; q < 3; ++q) S->pivot[q] = n ? s[q] / (double)n : 0.0;
    S->bad_input = s[3] != 0.0;
    S->done = S->bad_input || n == 0;
}

// The local plane of the map at combined-grid cell (ci, cj, ck): z - z0 = a (x - x0) + b (y - y0) + d, in double, over the
// centroids of the cell (x0, y0, z0) and of its 8 horizontal neighbours at the same k that are in the map (count >=
// min_points), summed in the order row j, j-1, j+1, each i-1, i, i+1.  True with the plane's unit normal
// n = (-a, -b, 1) / |.|; false when the cell is outside +-(2^20 - 2) in i or j (its neighbours would leave the key range) or
// +-(2^20 - 1) in k, is not in the map, has fewer than 3 such cells, or the 3 x 3 system is singular (det <= kRegFitCond *
// Suu * Sww * S1).  k_reg_step and the mesh's normals (mesh.cuh) both call it, so the two cannot drift apart.
__device__ __forceinline__ bool reg_fit(const uint64_t* __restrict__ res_keys, const float4* __restrict__ res_acc, uint32_t n_res,
                                        uint32_t min_points, int ci, int cj, int ck, double& x0, double& y0, double& z0,
                                        double& nx, double& ny, double& nz) {
    const int lim = (1 << 20) - 1;
    if (ci < -lim + 1 || ci > lim - 1 || cj < -lim + 1 || cj > lim - 1 || ck < -lim || ck > lim) return false;
    // One lower bound per row (a row's cells are consecutive keys); the cell's own row goes first, and without the cell
    // in the map there is no plane.
    uint64_t k0 = reg_key(ci - 1, cj, ck);
    uint32_t at = reg_lower_bound(res_keys, n_res, k0);
    float hx[3], hy[3], hz[3];
    uint32_t hit = 0;
#pragma unroll
    for (int di = 0; di < 3; ++di)
        if (at < n_res && res_keys[at] == k0 + (uint64_t)di) {
            const float4 a = res_acc[at++];
            if (__float_as_uint(a.w) >= min_points) {
                const float4 c = acc_centroid(a, make_uint4(0u, 0u, 0u, 0u));
                hx[di] = c.x; hy[di] = c.y; hz[di] = c.z;
                hit |= 1u << di;
            }
        }
    if (!(hit & 2u)) return false;
    x0 = hx[1]; y0 = hy[1]; z0 = hz[1];
    double Suu = 0, Suw = 0, Su = 0, Sww = 0, Sw = 0, S1 = 0, Suh = 0, Swh = 0, Sh = 0;
    auto add = [&](float fx, float fy, float fz) {
        const double u = (double)fx - x0, w = (double)fy - y0, h = (double)fz - z0;
        Suu += u * u; Suw += u * w; Su += u; Sww += w * w; Sw += w; S1 += 1.0;
        Suh += u * h; Swh += w * h; Sh += h;
    };
#pragma unroll
    for (int di = 0; di < 3; ++di)
        if (hit & (1u << di)) add(hx[di], hy[di], hz[di]);
#pragma unroll
    for (int dj = -1; dj <= 1; dj += 2) {
        k0 = reg_key(ci - 1, cj + dj, ck);
        at = reg_lower_bound(res_keys, n_res, k0);
#pragma unroll
        for (int di = 0; di < 3; ++di)
            if (at < n_res && res_keys[at] == k0 + (uint64_t)di) {
                const float4 a = res_acc[at++];
                if (__float_as_uint(a.w) >= min_points) {
                    const float4 c = acc_centroid(a, make_uint4(0u, 0u, 0u, 0u));
                    add(c.x, c.y, c.z);
                }
            }
    }
    if (S1 < 3.0) return false;
    const double c00 = Sww * S1 - Sw * Sw, c01 = Sw * Su - Suw * S1, c02 = Suw * Sw - Sww * Su;
    const double c11 = Suu * S1 - Su * Su, c12 = Su * Suw - Suu * Sw;
    const double det = Suu * c00 + Suw * c01 + Su * c02;
    if (!(det > kRegFitCond * Suu * Sww * S1)) return false;
    const double a = (c00 * Suh + c01 * Swh + c02 * Sh) / det;
    const double b = (c01 * Suh + c11 * Swh + c12 * Sh) / det;
    const double nn = sqrt(a * a + b * b + 1.0);
    nx = -a / nn; ny = -b / nn; nz = 1.0 / nn;
    return true;
}

// One Gauss-Newton linearisation: per CTA the sums of the normal equations over the point's correspondences.
__global__ void __launch_bounds__(kThreads) k_reg_step(const float4* __restrict__ pts, size_t n, const RegState* __restrict__ S,
                                                       RegParams P, const uint64_t* __restrict__ res_keys,
                                                       const float4* __restrict__ res_acc,
                                                       const uint32_t* __restrict__ n_res_ptr, double* __restrict__ part) {
    wait_prior();
    if (S->done) return;   // an earlier iteration of the call converged or failed: the queued rest exits here
    __shared__ double sm[kWarps];
    __shared__ double T[12], piv[3];
    if (threadIdx.x < 12) T[threadIdx.x] = S->T[threadIdx.x];
    if (threadIdx.x < 3) piv[threadIdx.x] = S->pivot[threadIdx.x];
    __syncthreads();
    const uint32_t n_res = *n_res_ptr;
    double H[21], g[6], cnt = 0.0, ss = 0.0;
#pragma unroll
    for (int q = 0; q < 21; ++q) H[q] = 0.0;
#pragma unroll
    for (int q = 0; q < 6; ++q) g[q] = 0.0;
    for (size_t idx = (size_t)blockIdx.x * kThreads + threadIdx.x; idx < n; idx += (size_t)gridDim.x * kThreads) {
        const float4 p = pts[idx];
        double x, y, z;
        reg_apply(T, p.x, p.y, p.z, x, y, z);
        int ci, cj, ck;
        combined_cell((float)x, (float)y, (float)z, P.inv_c, P.inv_cz, ci, cj, ck);
        // the hit cell's plane; without the hit cell in the map, or without a plane, the point has no correspondence
        double x0, y0, z0, nx, ny, nz;
        if (!reg_fit(res_keys, res_acc, n_res, P.min_points, ci, cj, ck, x0, y0, z0, nx, ny, nz)) continue;
        const double r = nx * (x - x0) + ny * (y - y0) + nz * (z - z0);
        if (!(fabs(r) <= P.max_distance)) continue;
        const double qx = x - piv[0], qy = y - piv[1], qz = z - piv[2];
        const double J[6] = {qy * nz - qz * ny, qz * nx - qx * nz, qx * ny - qy * nx, nx, ny, nz};
        int q = 0;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
#pragma unroll
            for (int j = i; j < 6; ++j) H[q++] += J[i] * J[j];
            g[i] += J[i] * r;
        }
        cnt += 1.0;
        ss += r * r;
    }
    double* out = part + (size_t)blockIdx.x * kRegSums;
#pragma unroll
    for (int q = 0; q < 21; ++q) { const double s = reg_block_sum(H[q], sm); if (threadIdx.x == 0) out[q] = s; }
#pragma unroll
    for (int q = 0; q < 6; ++q) { const double s = reg_block_sum(g[q], sm); if (threadIdx.x == 0) out[21 + q] = s; }
    { const double s = reg_block_sum(cnt, sm); if (threadIdx.x == 0) out[27] = s; }
    { const double s = reg_block_sum(ss, sm); if (threadIdx.x == 0) out[28] = s; }
}

// symmetric 6 x 6 eigen-decomposition by cyclic Jacobi rotations: A = V diag(w) V^T (A is destroyed)
__device__ void reg_eigen6(double (*A)[6], double (*V)[6], double* w) {
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) V[i][j] = (i == j);
    for (int sweep = 0; sweep < 50; ++sweep) {
        bool rotated = false;
        for (int p = 0; p < 5; ++p)
            for (int q = p + 1; q < 6; ++q) {
                const double apq = A[p][q];
                if (apq == 0.0) continue;
                if (fabs(apq) <= 1e-300 || fabs(apq) <= 1e-18 * (fabs(A[p][p]) + fabs(A[q][q]))) {
                    A[p][q] = A[q][p] = 0.0;
                    continue;
                }
                rotated = true;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
                for (int k = 0; k < 6; ++k) {
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - sn * akq;
                    A[k][q] = sn * akp + c * akq;
                }
                for (int k = 0; k < 6; ++k) {
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - sn * aqk;
                    A[q][k] = sn * apk + c * aqk;
                }
                for (int k = 0; k < 6; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - sn * vkq;
                    V[k][q] = sn * vkp + c * vkq;
                }
            }
        if (!rotated) break;
    }
    for (int i = 0; i < 6; ++i) w[i] = A[i][i];
}

// One CTA: adds the CTA partials in CTA order, solves, updates S->T and the stop flags.
__global__ void __launch_bounds__(kThreads) k_reg_solve(const double* __restrict__ part, uint32_t blocks, RegParams P,
                                                        uint32_t first, RegState* __restrict__ S) {
    wait_prior();
    __shared__ double tot[kRegSums];
    __shared__ double A[6][6], V[6][6], w[6], g[6], x[6];   // (thread 0's working set: shared, not a stack frame)
    if (S->done) return;
    // thread q < 29 adds quantity q over the CTAs, in CTA order
    if (threadIdx.x < 29) {
        double s = 0.0;
        for (uint32_t b = 0; b < blocks; ++b) s += part[(size_t)b * kRegSums + threadIdx.x];
        tot[threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    int q = 0;
    for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) { A[i][j] = A[j][i] = tot[q++]; }
    for (int i = 0; i < 6; ++i) g[i] = tot[21 + i];
    const double cnt = tot[27];
    const double rms = cnt > 0.0 ? sqrt(tot[28] / cnt) : 0.0;
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) S->info[i * 6 + j] = A[i][j];
    S->n_inliers = (uint32_t)cnt;
    if (first) S->rms_initial = rms;
    S->rms_final = rms;
    if (cnt < 6.0) {   // too few correspondences: T_init stands
        for (int i = 0; i < 12; ++i) S->T[i] = S->T0[i];
        S->rank = 0; S->converged = 0; S->done = 1;
        return;
    }
    S->iterations += 1;
    // rotations enter as arc lengths at the inliers' lever arm L (rotation block trace / translation block trace = mean
    // |q x n|^2), so that the six directions share one unit and degenerate_ratio compares like with like
    const double tr_r = A[0][0] + A[1][1] + A[2][2], tr_t = A[3][3] + A[4][4] + A[5][5];
    const double L = (tr_r > 0.0 && tr_t > 0.0) ? sqrt(tr_r / tr_t) : 1.0;
    double sc[6];
    for (int i = 0; i < 6; ++i) sc[i] = i < 3 ? 1.0 / L : 1.0;
    for (int i = 0; i < 6; ++i) {
        g[i] *= sc[i];
        for (int j = 0; j < 6; ++j) A[i][j] *= sc[i] * sc[j];
    }
    reg_eigen6(A, V, w);
    double wmax = 0.0;
    for (int i = 0; i < 6; ++i) wmax = fmax(wmax, w[i]);
    const double thr = P.degenerate_ratio * wmax;
    for (int i = 0; i < 6; ++i) x[i] = 0.0;
    uint32_t rank = 0;
    for (int e = 0; e < 6; ++e) {
        if (!(w[e] > 0.0) || w[e] < thr) continue;
        double d = 0.0;
        for (int i = 0; i < 6; ++i) d += V[i][e] * g[i];
        const double f = -d / w[e];
        for (int i = 0; i < 6; ++i) x[i] += f * V[i][e];
        ++rank;
    }
    for (int i = 0; i < 6; ++i) x[i] *= sc[i];
    S->rank = rank;
    // rotation about the pivot by the axis-angle x[0..3] (Rodrigues), then translation x[3..6]
    const double th = sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
    double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (th > 0.0) {
        const double kx = x[0] / th, ky = x[1] / th, kz = x[2] / th, c = cos(th), s = sin(th), v = 1.0 - c;
        R[0] = c + kx * kx * v;      R[1] = kx * ky * v - kz * s; R[2] = kx * kz * v + ky * s;
        R[3] = ky * kx * v + kz * s; R[4] = c + ky * ky * v;      R[5] = ky * kz * v - kx * s;
        R[6] = kz * kx * v - ky * s; R[7] = kz * ky * v + kx * s; R[8] = c + kz * kz * v;
    }
    const double* pv = S->pivot;
    double D[12];
    for (int i = 0; i < 3; ++i) {
        D[i * 4 + 0] = R[i * 3 + 0]; D[i * 4 + 1] = R[i * 3 + 1]; D[i * 4 + 2] = R[i * 3 + 2];
        D[i * 4 + 3] = pv[i] + x[3 + i] - (R[i * 3 + 0] * pv[0] + R[i * 3 + 1] * pv[1] + R[i * 3 + 2] * pv[2]);
    }
    double Tn[12];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 4; ++j) {
            double s = D[i * 4 + 0] * S->T[0 * 4 + j] + D[i * 4 + 1] * S->T[1 * 4 + j] + D[i * 4 + 2] * S->T[2 * 4 + j];
            if (j == 3) s += D[i * 4 + 3];
            Tn[i * 4 + j] = s;
        }
    for (int i = 0; i < 12; ++i) S->T[i] = Tn[i];
    const double tn = sqrt(x[3] * x[3] + x[4] * x[4] + x[5] * x[5]);
    if (th < P.min_rotation && tn < P.min_translation) { S->converged = 1; S->done = 1; }
}

}  // namespace o3r
