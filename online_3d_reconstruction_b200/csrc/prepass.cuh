// prepass.cuh — the per-frame reductions that run before the hot path (SURVEY §8f-3):
//   createPlaneFittedDisparityImages (pose_functions.cpp:900-985): per segment label, the normal equations of the
//     least-squares plane d = a*x + b*y + c over the label's pixels strictly inside the ROI (:929), and
//   getMean / getVariance (pose_functions.cpp:987-1028), the bad-frame gate (pose.cpp:187-196, :975-982).
// The nine sums of the normal equations are integers (x, y, 8-bit d), accumulated in u64: exact, so the 3x3 solve on the
// host sees the same numbers as the reference's double sums.  The variance sums are doubles; they are reduced per
// image row in a fixed tree order and the rows are added in order on the host (deterministic, not the reference's
// strictly sequential order, whose own rounding error over 748 000 additions is ~1e-12: agreement to 1e-10 relative is asserted).
#pragma once
#include "common.cuh"

namespace o3r {

constexpr int kLabSums = 10;   // total, n, Sx, Sy, Sxx, Sxy, Syy, Sxd, Syd, Sd

// grid: (row blocks), one CTA per 8 image rows; out[256][kLabSums] u64, zeroed by the caller
__global__ void __launch_bounds__(kThreads) k_label_sums(const uint8_t* __restrict__ labels, size_t lstep,
                                                         const uint8_t* __restrict__ disp, size_t dstep, int rows, int cols,
                                                         int x0, int bb, unsigned long long* __restrict__ out) {
    wait_prior();
    __shared__ unsigned long long acc[256 * kLabSums];
    for (int i = threadIdx.x; i < 256 * kLabSums; i += kThreads) acc[i] = 0ull;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int y0 = blockIdx.x * 8;
    for (int y = y0; y < min(y0 + 8, rows); ++y) {
        const bool yin = y > bb && y < rows - bb;   // strict (pose_functions.cpp:929)
        for (int xb = 0; xb < cols; xb += kThreads) {
            const int x = xb + threadIdx.x;
            const bool valid = x < cols;
            const unsigned vm = __ballot_sync(kFull, valid);
            if (!valid) continue;
            const unsigned l = labels[(size_t)y * lstep + x];
            const bool in = yin && x > x0 && x < cols - bb;
            const unsigned long long d = disp[(size_t)y * dstep + x];
            // one shared-memory atomic per distinct label of the warp (labels are large coherent regions)
            const unsigned peers = __match_any_sync(vm, l);
            const int leader = __ffs(peers) - 1;
            unsigned long long v[kLabSums];
            v[0] = 1ull;
            v[1] = in ? 1ull : 0ull;
            v[2] = in ? (unsigned long long)x : 0ull;
            v[3] = in ? (unsigned long long)y : 0ull;
            v[4] = in ? (unsigned long long)x * x : 0ull;
            v[5] = in ? (unsigned long long)x * y : 0ull;
            v[6] = in ? (unsigned long long)y * y : 0ull;
            v[7] = in ? (unsigned long long)x * d : 0ull;
            v[8] = in ? (unsigned long long)y * d : 0ull;
            v[9] = in ? d : 0ull;
            if (peers == kFull) {   // the whole (full) warp agrees: warp sums, one atomic per sum
#pragma unroll
                for (int q = 0; q < kLabSums; ++q) {
                    unsigned long long s = v[q];
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(vm, s, o);
                    v[q] = s;
                }
                if (lane == leader && l != 0)
#pragma unroll
                    for (int q = 0; q < kLabSums; ++q) atomicAdd(&acc[l * kLabSums + q], v[q]);
            } else if (l != 0) {
#pragma unroll
                for (int q = 0; q < kLabSums; ++q)
                    if (v[q]) atomicAdd(&acc[l * kLabSums + q], v[q]);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256 * kLabSums; i += kThreads)
        if (acc[i]) atomicAdd(&out[i], acc[i]);
}

// per ROI row: sum over valid samples of f(d) where f = d (pass 0) or (d - mean)^2 (pass 1).  One CTA per row,
// fixed-order tree reduction.  The sample is the u8 disparity, or the plane-fitted value of its label.
__global__ void __launch_bounds__(kThreads) k_row_moment(const uint8_t* __restrict__ disp, size_t dstep,
                                                         const uint8_t* __restrict__ labels, size_t lstep,
                                                         const double* __restrict__ coef, int n_planes, int cols, int x0,
                                                         int bb, double min_disp, int pass, double mean,
                                                         double* __restrict__ row_out) {
    wait_prior();
    __shared__ double sm[kThreads];
    const int y = bb + blockIdx.x;
    double s = 0.0;
    for (int x = x0 + threadIdx.x; x < cols - bb; x += kThreads) {
        double d;
        if (labels) {   // pose_functions.cpp:968-971 (label 0 and labels past the last plane stay 0.0)
            const int l = labels[(size_t)y * lstep + x];
            d = 0.0;
            if (l != 0 && l <= n_planes) {
                const double* c = coef + 3 * (l - 1);
                d = __dadd_rn(__dadd_rn(__dmul_rn(__dmul_rn(1.0, c[0]), (double)x), __dmul_rn(__dmul_rn(1.0, c[1]), (double)y)),
                              __dmul_rn(1.0, c[2]));
            }
        } else {
            d = (double)disp[(size_t)y * dstep + x];
        }
        if (d > min_disp) s = __dadd_rn(s, pass == 0 ? d : __dmul_rn(__dsub_rn(d, mean), __dsub_rn(d, mean)));
    }
    sm[threadIdx.x] = s;
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sm[threadIdx.x] = __dadd_rn(sm[threadIdx.x], sm[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) row_out[blockIdx.x] = sm[0];
}

}  // namespace o3r
