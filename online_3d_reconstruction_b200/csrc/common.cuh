// common.cuh — shared device helpers for the o3r CUDA library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "../../include/o3r.h"

namespace o3r {

constexpr int kThreads = 256;          // every kernel in this library runs 256-thread CTAs
constexpr int kWarps = kThreads / 32;
constexpr unsigned kFull = 0xffffffffu;

// Every __global__ of the library calls this first, before any global read, write or atomic.  The library launches its
// kernels with programmatic stream serialisation (LAUNCH_N, host_ctx.cuh): a kernel may be launched and its CTAs placed
// while the previous kernel on the stream is still draining, and this waits until that kernel has completed and its writes
// are visible.  Since every kernel waits here before it touches memory, stream order holds transitively.  No kernel
// triggers its dependents early, so what overlaps is the launch and the CTA rasterisation only.  (A no-op in a kernel
// launched without the attribute.)
__device__ __forceinline__ void wait_prior() { cudaGridDependencySynchronize(); }

// One frame's inputs as the kernels see them (device pointers).
struct FrameDev {
    const uint8_t* disp;
    const uint8_t* bgr;
    const uint8_t* labels;
    const double* plane_coef;
    const float* kp_xy;
    unsigned long long disp_step, bgr_step, labels_step;
    int n_planes, n_kp;
    float T[12];
};

// pcl::VoxelGrid per-cloud grid (SURVEY §8a row VG), computed on the device from the bbox.
struct GridParams {
    float inv[3];
    int min_b[3];
    int mul1, mul2;     // divb_mul_[1], divb_mul_[2]
    int passthrough;    // PCL's int32 overflow guard tripped: output = input
    int empty;
    int key_bits;       // live bits of the leaf index (= bits of div0*div1*div2 - 1)
};

// order-preserving float <-> uint mapping for atomicMin/atomicMax bbox reductions
__host__ __device__ __forceinline__ uint32_t f2ord(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float ord2f(uint32_t u) {
    u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}

// Exclusive scan of one value per thread over the 256-thread CTA. `sm` is 34 words of shared memory.
// Ends with a barrier so `sm` may be reused immediately.
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* sm, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < kWarps ? sm[lane] : 0u, winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(kFull, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < kWarps) sm[lane] = winc - w;
        if (lane == kWarps - 1) sm[33] = winc;
    }
    __syncthreads();
    total = sm[33];
    const uint32_t r = sm[warp] + inc - v;
    __syncthreads();
    return r;
}

// the rigid transform of pcl::transformPointCloud (float, left to right, no FMA) — SURVEY §8a row T
__device__ __forceinline__ void xform(const float* T, float x, float y, float z, float& ox, float& oy, float& oz) {
    ox = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[0], x), __fmul_rn(T[1], y)), __fmul_rn(T[2], z)), T[3]);
    oy = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[4], x), __fmul_rn(T[5], y)), __fmul_rn(T[6], z)), T[7]);
    oz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[8], x), __fmul_rn(T[9], y)), __fmul_rn(T[10], z)), T[11]);
}

// pcl::VoxelGrid leaf index (relative to min_b), PCL 1.8 voxel_grid.hpp first pass.  PCL computes it in int and lets it
// wrap when div0*div1*div2 exceeds INT32_MAX (see make_grid); uint32 arithmetic gives the same bits without the
// undefined signed overflow.
__device__ __forceinline__ uint32_t vg_rel_idx(const GridParams& G, float x, float y, float z) {
    const int i0 = (int)(__fsub_rn(floorf(__fmul_rn(x, G.inv[0])), (float)G.min_b[0]));
    const int i1 = (int)(__fsub_rn(floorf(__fmul_rn(y, G.inv[1])), (float)G.min_b[1]));
    const int i2 = (int)(__fsub_rn(floorf(__fmul_rn(z, G.inv[2])), (float)G.min_b[2]));
    return (uint32_t)i0 + (uint32_t)i1 * (uint32_t)G.mul1 + (uint32_t)i2 * (uint32_t)G.mul2;
}

// 64-bit absolute cell key: (k+2^20)<<42 | (j+2^20)<<21 | (i+2^20)
__device__ __forceinline__ uint64_t abs_cell_key(float x, float y, float z, float ix, float iy, float iz) {
    const long long B = 1 << 20;
    const long long i = (long long)floorf(__fmul_rn(x, ix));
    const long long j = (long long)floorf(__fmul_rn(y, iy));
    const long long k = (long long)floorf(__fmul_rn(z, iz));
    return ((uint64_t)(k + B) << 42) | ((uint64_t)(j + B) << 21) | (uint64_t)(i + B);
}

// GridParams from an ordered-uint bbox {minx,miny,minz,maxx,maxy,maxz} — PCL's guard + min_b/div_b
__device__ __forceinline__ GridParams make_grid(const uint32_t* bb, float ix, float iy, float iz) {
    GridParams G;
    G.inv[0] = ix; G.inv[1] = iy; G.inv[2] = iz;
    G.empty = (bb[0] == 0xffffffffu);   // untouched min => no points
    G.passthrough = 0;
    G.key_bits = 1;
    G.mul1 = G.mul2 = 0;
    G.min_b[0] = G.min_b[1] = G.min_b[2] = 0;
    if (G.empty) return G;
    float mn[3], mx[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) { mn[a] = ord2f(bb[a]); mx[a] = ord2f(bb[3 + a]); }
    const long long dx = (long long)(__fmul_rn(__fsub_rn(mx[0], mn[0]), ix)) + 1;
    const long long dy = (long long)(__fmul_rn(__fsub_rn(mx[1], mn[1]), iy)) + 1;
    const long long dz = (long long)(__fmul_rn(__fsub_rn(mx[2], mn[2]), iz)) + 1;
    if (dx * dy * dz > 2147483647ll) { G.passthrough = 1; return G; }
    int div[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        G.min_b[a] = (int)floorf(__fmul_rn(mn[a], G.inv[a]));
        const int max_b = (int)floorf(__fmul_rn(mx[a], G.inv[a]));
        div[a] = max_b - G.min_b[a] + 1;
    }
    G.mul1 = div[0];
    G.mul2 = (int)((uint32_t)div[0] * (uint32_t)div[1]);   // (wraps as PCL's int product does)
    const long long cells = (long long)div[0] * div[1] * div[2];
    // PCL's index is a 32-bit int: when div0*div1*div2 exceeds it (the guard above uses the slightly smaller d = (int64)((max - min) * inv) + 1)
    // the index wraps, here exactly as in PCL, and all 32 bits are live
    G.key_bits = cells > 1 ? min(32, 64 - __clzll(cells - 1)) : 1;
    return G;
}

}  // namespace o3r
