// blur.cuh — the blur step of createSingleImgPtCloud (pose_functions.cpp:1040-1047) for u8 disparity,
// with the two filters north_star names: exact k x k median (cv::medianBlur: BORDER_REPLICATE, odd k)
// and normalised box (cv::blur: anchor k/2, BORDER_REFLECT_101, round-half-even(S / k^2)).
//
// One CTA produces a block of 64 output columns x 128 rows (box) or 32 rows (median).  The input block with its halo is
// staged in shared memory once (the border rule is applied while staging); a thread (box) or a group of four lanes (median)
// walks one output row: a running sum, or a 256-bin histogram in shared memory through which the median is tracked, slid
// one column per step (k entries in, k out).  Outputs leave through a shared-memory tile so the global stores are row-coalesced.
#pragma once
#include "common.cuh"

namespace o3r {

constexpr int kBlurRows = 128;   // threads per CTA; output rows per CTA of the box filter (one thread per row)
constexpr int kBlurStrip = 64;   // output columns per CTA
constexpr int kBlurMaxK = 127;
constexpr int kMedLanes = 4;                        // median: lanes that share one output row's histogram
constexpr int kMedRows = kBlurRows / kMedLanes;     // median: output rows per CTA
constexpr int kMedStride = kMedRows + 1;            // histogram words of one bin pair, padded: a row's lanes hit different banks

struct BlurJob {
    const uint8_t* src; unsigned long long sstep;
    uint8_t* dst; unsigned long long dstep;
};

__host__ __device__ inline int blur_rows(int mode) { return mode == O3R_BLUR_MEDIAN ? kMedRows : kBlurRows; }
__host__ __device__ inline int blur_pitch(int k) {
    int w = kBlurStrip + k - 1;
    int p = (w + 3) / 4;
    if ((p & 1) == 0) ++p;  // odd number of words per row => the 32 rows of a warp hit 32 different banks
    return p * 4;
}
inline size_t blur_smem(int k, int mode) {
    const int rows = blur_rows(mode);
    size_t s = (size_t)(rows + k - 1) * blur_pitch(k) + (size_t)rows * kBlurStrip;
    s = (s + 15) & ~(size_t)15;
    if (mode == O3R_BLUR_MEDIAN) s += (size_t)128 * kMedStride * 4;   // 256 16-bit counters per output row, two to a word
    return s;
}

__device__ __forceinline__ int dev_reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = (i < 0) ? -i : 2 * n - 2 - i;
    return i;
}

template <int MODE>
__global__ void __launch_bounds__(kBlurRows) k_blur(const BlurJob* __restrict__ jobs, int rows, int cols, int k,
                                                    int rx0, int ry0, int rx1, int ry1) {
    wait_prior();
    extern __shared__ __align__(16) unsigned char bsm[];
    constexpr int ROWS = MODE == O3R_BLUR_MEDIAN ? kMedRows : kBlurRows;
    const BlurJob job = jobs[blockIdx.z];
    const int a = k / 2, pitch = blur_pitch(k);
    const int bx = rx0 + blockIdx.x * kBlurStrip, by = ry0 + blockIdx.y * ROWS;
    const int tw = kBlurStrip + k - 1, th = ROWS + k - 1;
    unsigned char* tin = bsm;
    unsigned char* tout = bsm + (size_t)th * pitch;
    const int tid = threadIdx.x;
    // stage input block + halo, border rule applied here
    for (int i = tid; i < tw * th; i += kBlurRows) {
        const int ly = i / tw, lx = i - ly * tw;
        int gy = by - a + ly, gx = bx - a + lx;
        if (MODE == O3R_BLUR_MEDIAN) {
            gy = min(max(gy, 0), rows - 1);
            gx = min(max(gx, 0), cols - 1);
        } else {
            gy = dev_reflect101(gy, rows);
            gx = dev_reflect101(gx, cols);
        }
        tin[ly * pitch + lx] = job.src[(size_t)gy * job.sstep + gx];
    }
    if (MODE == O3R_BLUR_MEDIAN) {
        // Huang's sliding median, one histogram per output row in shared memory: 256 16-bit counters, two to a word, laid out
        // [word][row] with a padded stride.  FOUR lanes share a row: each takes every fourth window row of the k values that
        // enter and the k that leave per step, so a step's dependent chain is a quarter as long, and the 16 KB of histograms
        // per CTA (instead of 64 KB with one thread per row) let 36 warps live on an SM instead of 8 — the first version of
        // this kernel sat at 12 % occupancy waiting for its own shared-memory round trips.  Counters move by shared-memory
        // atomics WITHOUT a result (nobody waits for them; lanes of one row may hit the same counter), unchanged columns are
        // skipped, and the median is tracked, not searched: `lt` counts the window's values below `med` (register
        // arithmetic per update, summed over the four lanes by two shuffles), and `med` walks to the bin where
        // lt <= k*k/2 < lt + count(med) — a step or two per pixel on real disparities; the four lanes do that walk redundantly
        // on the same counters.  16-bit halves never carry: a counter is decremented only for a value that was counted, and
        // k*k <= 127^2 < 65536.
        uint32_t* hist_all = reinterpret_cast<uint32_t*>(bsm + (((size_t)th * pitch + (size_t)ROWS * kBlurStrip + 15) & ~(size_t)15));
        for (int i = tid; i < 128 * kMedStride; i += kBlurRows) hist_all[i] = 0u;
        __syncthreads();
        const int row = tid / kMedLanes, sub = tid % kMedLanes;
        uint32_t* hist = hist_all + row;
        const unsigned char* myrow = tin + row * pitch;   // window rows are myrow + dy*pitch, dy in [0,k)
        for (int dy = sub; dy < k; dy += kMedLanes) {
            const unsigned char* r = myrow + dy * pitch;
#pragma unroll 4
            for (int dx = 0; dx < k; ++dx) {
                const int v = r[dx];
                atomicAdd(&hist[(v >> 1) * kMedStride], 1u << ((v & 1) << 4));
            }
        }
        const int half = (k * k) / 2;
        int med = 0, lt = 0;
        for (int x = 0; x < kBlurStrip; ++x) {
            int d = 0;
            if (x > 0) {
                const unsigned char* r = myrow + x - 1;
#pragma unroll 4
                for (int dy = sub; dy < k; dy += kMedLanes) {
                    const int vo = r[dy * pitch], vn = r[dy * pitch + k];
                    if (vo != vn) {
                        atomicSub(&hist[(vo >> 1) * kMedStride], 1u << ((vo & 1) << 4));
                        atomicAdd(&hist[(vn >> 1) * kMedStride], 1u << ((vn & 1) << 4));
                        d += (vn < med ? 1 : 0) - (vo < med ? 1 : 0);
                    }
                }
            }
            d += __shfl_xor_sync(kFull, d, 1);
            d += __shfl_xor_sync(kFull, d, 2);
            lt += d;
            __syncwarp();   // the row's counters are final for this step
            while (lt > half) {
                --med;
                lt -= (int)((hist[(med >> 1) * kMedStride] >> ((med & 1) << 4)) & 0xffffu);
            }
            for (;;) {
                const int c = (int)((hist[(med >> 1) * kMedStride] >> ((med & 1) << 4)) & 0xffffu);
                if (lt + c > half) break;
                lt += c;
                ++med;
            }
            if (sub == 0) tout[row * kBlurStrip + x] = (unsigned char)med;
            __syncwarp();   // every lane has read the counters before the next step moves them
        }
    } else {
        __syncthreads();
        const unsigned char* myrow = tin + tid * pitch;   // window rows are myrow + dy*pitch, dy in [0,k)
        const int kk = k * k;
        int S = 0;
        for (int dy = 0; dy < k; ++dy)
            for (int dx = 0; dx < k; ++dx) S += myrow[dy * pitch + dx];
        for (int x = 0; x < kBlurStrip; ++x) {
            if (x > 0)
                for (int dy = 0; dy < k; ++dy) S += (int)myrow[dy * pitch + x + k - 1] - (int)myrow[dy * pitch + x - 1];
            int q = S / kk;
            const int rem = S - q * kk;
            if (2 * rem > kk) q += 1;
            else if (2 * rem == kk) q += (q & 1);
            tout[tid * kBlurStrip + x] = (unsigned char)min(q, 255);
        }
    }
    __syncthreads();
    for (int i = tid; i < ROWS * kBlurStrip; i += kBlurRows) {
        const int ly = i / kBlurStrip, lx = i - ly * kBlurStrip;
        const int gy = by + ly, gx = bx + lx;
        if (gy < ry1 && gx < rx1) job.dst[(size_t)gy * job.dstep + gx] = tout[i];
    }
}

// ---- cv::bilateralFilter(u8, d = k, sigmaColor = 2k, sigmaSpace = k/2): the reference's LIVE blur (pose_functions.cpp:1044)
// OpenCV 3.1 bilateralFilter_8u: BORDER_REFLECT_101 halo, circular tap mask of radius k/2 walked row-major, weight =
// space_weight[tap] * color_weight[|v - v0|] (float LUTs computed on the host with std::exp, exactly like OpenCV
// and the oracle do), two sequential float accumulations per pixel, round-half-even(sum / wsum).  No FMA: the products
// and sums are rounded one by one in the tap order, so the result equals the CPU loop bit for bit.
// One CTA = 32 x 8 threads, each producing kBilPX horizontally adjacent outputs; the tile + halo, both LUTs and the per-row
// tap extents sit in shared memory (the colour LUT is read at data-dependent indices: shared memory, not constant memory).
// The kernel lives on the shared-memory pipe and on instruction issue together (709 taps per pixel at k = 30), so a thread
// shares what its two pixels have in common: the byte at column x + t of a window row is tap j = t of pixel x and tap j = t - 1
// of pixel x + 1, and its space weight for the second pixel is the one loaded a step earlier.  Per step: ONE byte load, ONE
// byte -> float conversion and ONE space-weight load serve both pixels; each pixel adds its colour-weight load (LUT mirrored
// around entry 255: cw[255 + v - v0], one scaled add away from the byte), two products and two sums — in exactly the tap
// order of the scalar loop, pixel by pixel.
constexpr int kBilTX = 32, kBilTY = 8, kBilPX = 2, kBilW = kBilTX * kBilPX;

struct BilateralLut {       // device copies, built once per context
    const float* color_w;   // [256]
    const float* space_w;   // [maxk] in tap order
    const int* jmax;        // [2 * radius + 1]: taps of row i are j in [-jmax, jmax]
    int radius, maxk;
};

inline size_t bilateral_smem(int radius, int maxk) {
    const int tw = kBilW + 2 * radius, th = kBilTY + 2 * radius;
    size_t s = ((size_t)tw * th + 15) & ~(size_t)15;
    return s + (size_t)512 * 4 + (size_t)maxk * 4 + (size_t)(2 * radius + 1) * 4;
}

__global__ void __launch_bounds__(kBilTX * kBilTY) k_bilateral(const BlurJob* __restrict__ jobs, BilateralLut L, int rows,
                                                               int cols, int rx0, int ry0, int rx1, int ry1) {
    wait_prior();
    extern __shared__ __align__(16) unsigned char bsm[];
    const BlurJob job = jobs[blockIdx.z];
    const int r = L.radius, tw = kBilW + 2 * r, th = kBilTY + 2 * r;
    unsigned char* tin = bsm;
    float* cw = reinterpret_cast<float*>(bsm + (((size_t)tw * th + 15) & ~(size_t)15));
    float* sw = cw + 512;
    int* jm = reinterpret_cast<int*>(sw + L.maxk);
    const int tid = threadIdx.y * kBilTX + threadIdx.x, nthr = kBilTX * kBilTY;
    const int bx = rx0 + blockIdx.x * kBilW, by = ry0 + blockIdx.y * kBilTY;
    for (int i = tid; i < tw * th; i += nthr) {
        const int ly = i / tw, lx = i - ly * tw;
        tin[i] = job.src[(size_t)dev_reflect101(by - r + ly, rows) * job.sstep + dev_reflect101(bx - r + lx, cols)];
    }
    for (int i = tid; i < 511; i += nthr) cw[i] = L.color_w[abs(i - 255)];
    for (int i = tid; i < L.maxk; i += nthr) sw[i] = L.space_w[i];
    for (int i = tid; i < 2 * r + 1; i += nthr) jm[i] = L.jmax[i];
    __syncthreads();
    const int gx = bx + threadIdx.x * kBilPX, gy = by + threadIdx.y;
    if (gx >= rx1 || gy >= ry1) return;
    const unsigned char* c0 = tin + (threadIdx.y + r) * tw + threadIdx.x * kBilPX + r;   // centre of the thread's first pixel
    const uint32_t cw_s = (uint32_t)__cvta_generic_to_shared(cw);
    uint32_t cw0 = cw_s + (uint32_t)(255 - (int)c0[0]) * 4u, cw1 = cw_s + (uint32_t)(255 - (int)c0[1]) * 4u;   // &cw[255 - v0]
    asm volatile("" : "+r"(cw0), "+r"(cw1));   // opaque: keeps the per-tap address ONE scaled add (base + 4 v) instead of two
    auto cwv = [](uint32_t base, int v) {
        float w;
        asm("ld.shared.f32 %0, [%1];" : "=f"(w) : "r"(base + (uint32_t)v * 4u));
        return w;
    };
    float sum0 = 0.f, wsum0 = 0.f, sum1 = 0.f, wsum1 = 0.f;
    int k = 0;
    for (int i = -r; i <= r; ++i) {
        const int m = jm[i + r];
        const unsigned char* row = c0 + i * tw;
        const float* swr = sw + k + m;   // space weight of tap (i, j): swr[j]
        // the byte at column t is tap j = t of the first pixel and tap j = t - 1 of the second
        int v = row[-m];
        float sp = swr[-m];
        {   // t = -m: the first pixel's first tap
            const float w = __fmul_rn(sp, cwv(cw0, v));
            sum0 = __fadd_rn(sum0, __fmul_rn((float)v, w));
            wsum0 = __fadd_rn(wsum0, w);
        }
#pragma unroll 4
        for (int t = -m + 1; t <= m; ++t) {
            v = row[t];
            const float f = (float)v, s = swr[t];
            const float wa = __fmul_rn(s, cwv(cw0, v));
            sum0 = __fadd_rn(sum0, __fmul_rn(f, wa));
            wsum0 = __fadd_rn(wsum0, wa);
            const float wb = __fmul_rn(sp, cwv(cw1, v));
            sum1 = __fadd_rn(sum1, __fmul_rn(f, wb));
            wsum1 = __fadd_rn(wsum1, wb);
            sp = s;
        }
        {   // t = m + 1: the second pixel's last tap
            v = row[m + 1];
            const float w = __fmul_rn(sp, cwv(cw1, v));
            sum1 = __fadd_rn(sum1, __fmul_rn((float)v, w));
            wsum1 = __fadd_rn(wsum1, w);
        }
        k += 2 * m + 1;
    }
    uint8_t* out = job.dst + (size_t)gy * job.dstep + gx;
    out[0] = (unsigned char)__float2int_rn(__fdiv_rn(sum0, wsum0));
    if (gx + 1 < rx1) out[1] = (unsigned char)__float2int_rn(__fdiv_rn(sum1, wsum1));
}

}  // namespace o3r
