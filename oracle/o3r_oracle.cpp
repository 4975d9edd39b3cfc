/*
 * o3r_oracle.cpp — CPU restatement of the reference hot path.  TEST INFRASTRUCTURE ONLY
 * (see o3r_oracle.h).  Plain C++17, no dependencies.  Must be compiled with -ffp-contract=off.
 *
 * Parity status: the reference ships no tests and cannot be built here (PCL/OpenCV/Boost/VTK
 * absent), so this restatement is pinned only by the artefacts the reference ships
 * (tests/golden/, tests/test_oracle_golden.py): valid-pixel counts and variances from
 * build/output/log.txt, the medianBlurred_*.png outputs, the ordering/lattice of build/cloud.ply
 * and the author's B.png known-answer frame.  PCL/OpenCV internals are restated from memory of the
 * libraries' sources: formally "parity unpinned" for those internals (DESIGN.md §Oracle).
 */
#include "o3r_oracle.h"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

namespace {

inline int reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) {
        if (i < 0) i = -i;
        else i = 2 * n - 2 - i;
    }
    return i;
}
inline int clampi(int i, int lo, int hi) { return i < lo ? lo : (i > hi ? hi : i); }

/* cv::medianBlur(u8, k): exact median of the k x k window, BORDER_REPLICATE (SURVEY §8a row F). */
void median_u8(const uint8_t* src, size_t sstep, int rows, int cols, int k, uint8_t* dst, size_t dstep) {
    const int r = k / 2, half = (k * k) / 2;
    std::vector<int> hist(256);
    for (int y = 0; y < rows; ++y) {
        std::fill(hist.begin(), hist.end(), 0);
        for (int dy = -r; dy <= r; ++dy) {
            const uint8_t* row = src + (size_t)clampi(y + dy, 0, rows - 1) * sstep;
            for (int dx = -r; dx <= r; ++dx) hist[row[clampi(dx, 0, cols - 1)]]++;
        }
        for (int x = 0; x < cols; ++x) {
            if (x > 0) {
                const int xo = clampi(x - 1 - r, 0, cols - 1), xn = clampi(x + r, 0, cols - 1);
                for (int dy = -r; dy <= r; ++dy) {
                    const uint8_t* row = src + (size_t)clampi(y + dy, 0, rows - 1) * sstep;
                    hist[row[xo]]--;
                    hist[row[xn]]++;
                }
            }
            int acc = 0, v = 0;
            for (; v < 256; ++v) {
                acc += hist[v];
                if (acc > half) break;
            }
            dst[(size_t)y * dstep + x] = (uint8_t)v;
        }
    }
}

/* cv::blur(u8, Size(k,k)): anchor k/2, BORDER_REFLECT_101, integer sum, round-half-even(S/k^2). */
void box_u8(const uint8_t* src, size_t sstep, int rows, int cols, int k, uint8_t* dst, size_t dstep) {
    const int a = k / 2, kk = k * k;
    std::vector<int> colsum(cols);
    for (int y = 0; y < rows; ++y) {
        std::fill(colsum.begin(), colsum.end(), 0);
        for (int dy = 0; dy < k; ++dy) {
            const uint8_t* row = src + (size_t)reflect101(y - a + dy, rows) * sstep;
            for (int x = 0; x < cols; ++x) colsum[x] += row[x];
        }
        for (int x = 0; x < cols; ++x) {
            int S = 0;
            for (int dx = 0; dx < k; ++dx) S += colsum[reflect101(x - a + dx, cols)];
            int q = S / kk, rem = S % kk;
            if (2 * rem > kk) q += 1;
            else if (2 * rem == kk) q += (q & 1);
            dst[(size_t)y * dstep + x] = (uint8_t)(q > 255 ? 255 : q);
        }
    }
}

/* cv::bilateralFilter(u8, d, sigmaColor, sigmaSpace), OpenCV 3.1.0 modules/imgproc/src/smooth.cpp bilateralFilter_8u
 * (third-party, not under /root/reference; call site pose_functions.cpp:1044 with d = k, sigmaColor = 2k,
 * sigmaSpace = k/2 in integer division).  BORDER_REFLECT_101 halo, circular tap mask in row-major (i, j) order,
 * float LUTs (float)std::exp(.), per pixel two sequential float accumulations (the 3.1 SSE path vectorises across
 * pixels, so each pixel still sums its taps in this order), cvRound(sum / wsum) = round-half-even.  cn = 1 or 3. */
void bilateral_u8(const uint8_t* src, size_t sstep, int rows, int cols, int cn, int d, double sigma_color,
                  double sigma_space, uint8_t* dst, size_t dstep) {
    if (sigma_color <= 0) sigma_color = 1;
    if (sigma_space <= 0) sigma_space = 1;
    const double gauss_color_coeff = -0.5 / (sigma_color * sigma_color);
    const double gauss_space_coeff = -0.5 / (sigma_space * sigma_space);
    int radius = d <= 0 ? (int)std::lrint(sigma_space * 1.5) : d / 2;
    radius = radius < 1 ? 1 : radius;
    std::vector<float> color_weight((size_t)cn * 256);
    for (int i = 0; i < 256 * cn; ++i) color_weight[i] = (float)std::exp(i * i * gauss_color_coeff);
    std::vector<float> sw;
    std::vector<int> oi, oj;
    for (int i = -radius; i <= radius; ++i)
        for (int j = -radius; j <= radius; ++j) {
            const double r = std::sqrt((double)i * i + (double)j * j);
            if (r > radius) continue;
            sw.push_back((float)std::exp(r * r * gauss_space_coeff));
            oi.push_back(i); oj.push_back(j);
        }
    const size_t maxk = sw.size();
    for (int y = 0; y < rows; ++y)
        for (int x = 0; x < cols; ++x) {
            const uint8_t* c0 = src + (size_t)y * sstep + (size_t)x * cn;
            if (cn == 1) {
                float sum = 0.f, wsum = 0.f;
                const int val0 = c0[0];
                for (size_t k = 0; k < maxk; ++k) {
                    const int val = src[(size_t)reflect101(y + oi[k], rows) * sstep + reflect101(x + oj[k], cols)];
                    const float w = sw[k] * color_weight[std::abs(val - val0)];
                    sum += val * w;
                    wsum += w;
                }
                dst[(size_t)y * dstep + x] = (uint8_t)std::lrintf(sum / wsum);
            } else {
                float sb = 0.f, sg = 0.f, sr = 0.f, wsum = 0.f;
                const int b0 = c0[0], g0 = c0[1], r0 = c0[2];
                for (size_t k = 0; k < maxk; ++k) {
                    const uint8_t* q = src + (size_t)reflect101(y + oi[k], rows) * sstep + (size_t)reflect101(x + oj[k], cols) * 3;
                    const int b = q[0], g = q[1], r = q[2];
                    const float w = sw[k] * color_weight[std::abs(b - b0) + std::abs(g - g0) + std::abs(r - r0)];
                    sb += b * w; sg += g * w; sr += r * w;
                    wsum += w;
                }
                wsum = 1.f / wsum;
                uint8_t* o = dst + (size_t)y * dstep + (size_t)x * 3;
                o[0] = (uint8_t)std::lrintf(sb * wsum); o[1] = (uint8_t)std::lrintf(sg * wsum); o[2] = (uint8_t)std::lrintf(sr * wsum);
            }
        }
}


/* ---- pcl::StatisticalOutlierRemoval<PointXYZRGB> (PCL 1.8 filters/impl/statistical_outlier_removal.hpp; third-party, not
 * under /root/reference; call site pose_functions.cpp:1673-1686 with setMeanK(50), setStddevMulThresh(1.0)) -------------
 * For every point: nearestKSearch(point, mean_k + 1) on a pcl::KdTreeFLANN (exact search, flann::L2_Simple<float>:
 * d2 = ((dx*dx) + (dy*dy)) + (dz*dz) in float); dist_i = (float)(sum_{k=1..mean_k} sqrt((double)d2_k) / mean_k), k = 0 being
 * the query itself; then mean / stddev of dist over all points in double (sum, sq_sum += dist*dist with a float product),
 * variance = (sq_sum - sum*sum/n) / (n - 1), threshold = mean + mul * stddev; a point is REMOVED iff dist > threshold.
 * Restated from memory of the PCL sources ("parity unpinned"): the unqualified sqrt() is taken as the double overload and
 * a cloud with fewer than mean_k + 1 points (where PCL reads past the returned neighbours) sums what exists.
 * The k-NN itself is exact, so how it is found does not matter: here a uniform grid whose cube around the query grows
 * until the (mean_k+1)-th smallest distance is provably inside it; orc_sor(..., brute = 1) checks every pair instead. */
struct SorHeap {   /* max-heap of the smallest `cap` squared distances seen */
    std::vector<float> h; size_t cap;
    explicit SorHeap(size_t c) : cap(c) { h.reserve(c); }
    void clear() { h.clear(); }
    void push(float d) {
        if (h.size() < cap) { h.push_back(d); std::push_heap(h.begin(), h.end()); }
        else if (d < h.front()) { std::pop_heap(h.begin(), h.end()); h.back() = d; std::push_heap(h.begin(), h.end()); }
    }
};
inline float sor_d2(const o3r_point& a, const o3r_point& b) {
    const float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z;
    return ((dx * dx) + (dy * dy)) + (dz * dz);
}
inline float sor_mean_dist(SorHeap& H, int mean_k) {
    std::sort(H.h.begin(), H.h.end());   /* ascending: k = 0 (the query, 0.0) first */
    double sum = 0.0;
    for (size_t k = 1; k < H.h.size(); ++k) sum += std::sqrt((double)H.h[k]);
    return (float)(sum / mean_k);
}

void sor_distances(const o3r_point* pts, size_t n, int mean_k, int threads, bool brute, float* dist) {
    const size_t K = (size_t)mean_k + 1;
    if (n == 0) return;
    if (brute || n <= K) {
        auto work = [&](size_t lo, size_t hi) {
            SorHeap H(K);
            for (size_t i = lo; i < hi; ++i) {
                H.clear();
                for (size_t j = 0; j < n; ++j) H.push(sor_d2(pts[i], pts[j]));
                dist[i] = sor_mean_dist(H, mean_k);
            }
        };
        std::vector<std::thread> th;
        const int T = std::max(1, threads);
        for (int t = 0; t < T; ++t) th.emplace_back(work, n * t / T, n * (t + 1) / T);
        for (auto& x : th) x.join();
        return;
    }
    /* uniform grid: cell size from the density of a surface-like cloud, enlarged until the tables stay small */
    float mn[3] = {pts[0].x, pts[0].y, pts[0].z}, mx[3] = {pts[0].x, pts[0].y, pts[0].z};
    for (size_t i = 1; i < n; ++i) {
        const float v[3] = {pts[i].x, pts[i].y, pts[i].z};
        for (int a = 0; a < 3; ++a) { mn[a] = std::min(mn[a], v[a]); mx[a] = std::max(mx[a], v[a]); }
    }
    double ext[3] = {(double)mx[0] - mn[0], (double)mx[1] - mn[1], (double)mx[2] - mn[2]};
    double e[3] = {ext[0], ext[1], ext[2]};
    std::sort(e, e + 3);
    const double area = std::max(e[2] * e[1], 1e-12);
    double c = std::sqrt((double)K * area / (3.141592653589793 * (double)n));
    c = std::max(c, 1e-6);
    long long nc[3];
    for (;;) {
        for (int a = 0; a < 3; ++a) nc[a] = (long long)(ext[a] / c) + 2;
        if (nc[0] * nc[1] * nc[2] <= (1ll << 31) && nc[1] * nc[2] <= (1ll << 22)) break;
        c *= 1.26;
    }
    const double inv = 1.0 / c;
    auto cell = [&](const o3r_point& p, long long ijk[3]) {
        const float v[3] = {p.x, p.y, p.z};
        for (int a = 0; a < 3; ++a) ijk[a] = std::min<long long>(nc[a] - 1, std::max<long long>(0, (long long)std::floor(((double)v[a] - mn[a]) * inv)));
    };
    std::vector<std::pair<long long, uint32_t>> order(n);
    for (size_t i = 0; i < n; ++i) {
        long long ijk[3];
        cell(pts[i], ijk);
        order[i] = {ijk[0] + nc[0] * (ijk[1] + nc[1] * ijk[2]), (uint32_t)i};
    }
    std::sort(order.begin(), order.end());
    const size_t rows = (size_t)(nc[1] * nc[2]);
    std::vector<uint32_t> rb(rows + 1, 0);
    for (size_t i = 0; i < n; ++i) rb[(size_t)(order[i].first / nc[0]) + 1]++;
    for (size_t r = 0; r < rows; ++r) rb[r + 1] += rb[r];
    auto work = [&](size_t lo, size_t hi) {
        SorHeap H(K);
        for (size_t i = lo; i < hi; ++i) {
            long long q[3];
            cell(pts[i], q);
            for (long long s = 1;; ++s) {
                H.clear();
                for (long long dz = -s; dz <= s; ++dz)
                    for (long long dy = -s; dy <= s; ++dy) {
                        const long long y = q[1] + dy, z = q[2] + dz;
                        if (y < 0 || y >= nc[1] || z < 0 || z >= nc[2]) continue;
                        const size_t r = (size_t)(y + nc[1] * z);
                        const long long k0 = std::max<long long>(0, q[0] - s) + nc[0] * (long long)r,
                                        k1 = std::min<long long>(nc[0] - 1, q[0] + s) + nc[0] * (long long)r;
                        auto b = std::lower_bound(order.begin() + rb[r], order.begin() + rb[r + 1], std::make_pair(k0, 0u));
                        for (; b != order.begin() + rb[r + 1] && b->first <= k1; ++b) H.push(sor_d2(pts[i], pts[b->second]));
                    }
                const bool all = q[0] - s <= 0 && q[0] + s >= nc[0] - 1 && q[1] - s <= 0 && q[1] + s >= nc[1] - 1 &&
                                 q[2] - s <= 0 && q[2] + s >= nc[2] - 1;
                /* every point outside the cube is farther than (s - 0.05) cells (the margin covers the cell rounding) */
                const double reach = (s - 0.05) * c;
                if (all || (H.h.size() == K && (double)H.h.front() <= reach * reach)) break;
            }
            dist[i] = sor_mean_dist(H, mean_k);
        }
    };
    std::vector<std::thread> th;
    const int T = std::max(1, threads);
    for (int t = 0; t < T; ++t) th.emplace_back(work, n * t / T, n * (t + 1) / T);
    for (auto& x : th) x.join();
}

struct DispReader {
    const o3r_params* p;
    const o3r_frame* f;
    int type;
    const uint8_t* blurred = nullptr;
    size_t blurred_step = 0;
    /* pose_functions.cpp:1098-1104 (+ :1064-1068): the disparity value as a double */
    inline double at(int y, int x) const {
        if (blurred) return (double)blurred[(size_t)y * blurred_step + x];
        if (p->use_segment_labels && f->labels && f->plane_coef) {
            /* pose_functions.cpp:968-971: label l (1-based) -> 1.0*a*x + 1.0*b*y + 1.0*c; label 0 stays 0 */
            const int l = f->labels[(size_t)y * f->labels_step + x];
            if (l == 0 || l > f->n_planes) return 0.0;
            const double* c = f->plane_coef + 3 * (l - 1);
            return 1.0 * c[0] * x + 1.0 * c[1] * y + 1.0 * c[2];
        }
        const uint8_t* row = (const uint8_t*)f->disp + (size_t)y * f->disp_step;
        switch (type) {
            case O3R_DISP_U8: return (double)row[x];
            case O3R_DISP_U16: return (double)((const uint16_t*)row)[x] / p->disp_divisor;
            case O3R_DISP_F32: return (double)((const float*)row)[x];
            default: return ((const double*)row)[x];
        }
    }
};

/* pose_functions.cpp:1073-1084 / :1110-1121: Q*[x y d 1]^T (cv::Mat_<double> 4x4 * 4x1: each row summed
 * left to right), vec /= vec(3) (OpenCV: multiply by 1.0/s), float casts, BGR -> 0x00RRGGBB. */
inline o3r_point reproject(const o3r_params* p, const o3r_frame* f, int x, int y, double d) {
    const double* Q = p->Q;
    const double dx = (double)x, dy = (double)y;
    const double v0 = Q[0] * dx + Q[1] * dy + Q[2] * d + Q[3] * 1.0;
    const double v1 = Q[4] * dx + Q[5] * dy + Q[6] * d + Q[7] * 1.0;
    const double v2 = Q[8] * dx + Q[9] * dy + Q[10] * d + Q[11] * 1.0;
    const double v3 = Q[12] * dx + Q[13] * dy + Q[14] * d + Q[15] * 1.0;
    const double s = 1.0 / v3;
    o3r_point pt;
    pt.x = (float)(v0 * s);
    pt.y = (float)(v1 * s);
    pt.z = (float)(v2 * s);
    const uint8_t* c = f->bgr + (size_t)y * f->bgr_step + 3 * (size_t)x;
    pt.rgb = ((uint32_t)c[2] << 16) | ((uint32_t)c[1] << 8) | (uint32_t)c[0];
    return pt;
}

inline void mat4_mul(const float* a, const float* b, float* o) {
    float t[16];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            float s = a[i * 4 + 0] * b[0 * 4 + j];
            s = s + a[i * 4 + 1] * b[1 * 4 + j];
            s = s + a[i * 4 + 2] * b[2 * 4 + j];
            s = s + a[i * 4 + 3] * b[3 * 4 + j];
            t[i * 4 + j] = s;
        }
    std::memcpy(o, t, sizeof(t));
}

/* symmetric 3x3 eigen-decomposition by cyclic Jacobi (for cv::invert(..., DECOMP_SVD) of AtA) */
void jacobi3(double A[3][3], double V[3][3], double w[3]) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) V[i][j] = (i == j);
    for (int sweep = 0; sweep < 64; ++sweep) {
        double off = std::fabs(A[0][1]) + std::fabs(A[0][2]) + std::fabs(A[1][2]);
        if (off == 0.0) break;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                if (A[p][q] == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 3; ++k) {
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - s * akq;
                    A[k][q] = s * akp + c * akq;
                }
                for (int k = 0; k < 3; ++k) {
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - s * aqk;
                    A[q][k] = s * apk + c * aqk;
                }
                for (int k = 0; k < 3; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - s * vkq;
                    V[k][q] = s * vkp + c * vkq;
                }
            }
    }
    for (int i = 0; i < 3; ++i) w[i] = A[i][i];
}

}  // namespace

extern "C" {

int orc_blur_u8(const uint8_t* src, size_t src_step, int rows, int cols, int kernel, int mode,
                uint8_t* dst, size_t dst_step) {
    if (!src || !dst || rows <= 0 || cols <= 0 || kernel < 1) return O3R_ERR_INVALID;
    if (mode == O3R_BLUR_MEDIAN) {
        if ((kernel & 1) == 0) return O3R_ERR_INVALID; /* cv::medianBlur asserts on even ksize */
        median_u8(src, src_step, rows, cols, kernel, dst, dst_step);
    } else if (mode == O3R_BLUR_BOX) {
        box_u8(src, src_step, rows, cols, kernel, dst, dst_step);
    } else if (mode == O3R_BLUR_BILATERAL) { /* pose_functions.cpp:1044: bilateralFilter(src, dst, k, k*2, k/2) */
        bilateral_u8(src, src_step, rows, cols, 1, kernel, (double)(kernel * 2), (double)(kernel / 2), dst, dst_step);
    } else {
        return O3R_ERR_INVALID;
    }
    return O3R_OK;
}

int orc_bilateral_u8(const uint8_t* src, size_t src_step, int rows, int cols, int cn, int d, double sigma_color,
                     double sigma_space, uint8_t* dst, size_t dst_step) {
    if (!src || !dst || rows <= 0 || cols <= 0 || (cn != 1 && cn != 3)) return O3R_ERR_INVALID;
    bilateral_u8(src, src_step, rows, cols, cn, d, sigma_color, sigma_space, dst, dst_step);
    return O3R_OK;
}

int orc_create_single_img_pt_cloud(const o3r_params* p, const o3r_frame* f, int disp_type,
                                   o3r_point* out, size_t cap, size_t* n_out,
                                   uint8_t* mask, size_t mask_cap, size_t* n_scanned) {
    if (!p || !f || !n_out) return O3R_ERR_INVALID;
    const int rows = p->rows, cols = p->cols, x0 = p->cols_start_aft_cutout, bb = p->bounding_box;
    const int J = p->jump_pixels;
    DispReader rd{p, f, disp_type};
    std::vector<uint8_t> blurred;
    if (p->blur_kernel > 1) { /* pose_functions.cpp:1040-1047 */
        if (disp_type != O3R_DISP_U8 || p->use_segment_labels) return O3R_ERR_INVALID; /* cv rejects CV_64F */
        blurred.resize((size_t)rows * cols);
        int rc = orc_blur_u8((const uint8_t*)f->disp, f->disp_step, rows, cols, p->blur_kernel, p->blur_mode,
                             blurred.data(), (size_t)cols);
        if (rc) return rc;
        rd.blurred = blurred.data();
        rd.blurred_step = (size_t)cols;
    }
    size_t n = 0, ns = 0;
    int rc = O3R_OK;
    if (J != 1) { /* pose_functions.cpp:1057-1091 keypoints first, ORB order, int truncation */
        for (int i = 0; i < f->n_kp; ++i) {
            const int x = (int)f->kp_xy[2 * i], y = (int)f->kp_xy[2 * i + 1];
            if (x >= x0 && x < cols - bb && y >= bb && y < rows - bb) {
                const double d = rd.at(y, x);
                if (d > p->min_disparity) {
                    if (n < cap && out) out[n] = reproject(p, f, x, y, d);
                    else if (out) rc = O3R_ERR_CAPACITY;
                    ++n;
                }
            }
        }
    }
    if (J > 0) { /* pose_functions.cpp:1092-1130 */
        for (int y = bb; y < rows - bb; y += J)
            for (int x = x0; x < cols - bb; x += J) {
                const double d = rd.at(y, x);
                const bool valid = d > p->min_disparity;
                if (mask && ns < mask_cap) mask[ns] = valid ? 1 : 0;
                ++ns;
                if (valid) {
                    if (n < cap && out) out[n] = reproject(p, f, x, y, d);
                    else if (out) rc = O3R_ERR_CAPACITY;
                    ++n;
                }
            }
    }
    *n_out = n;
    if (n_scanned) *n_scanned = ns;
    return rc;
}

void orc_transform_pt_cloud(const o3r_point* in, size_t n, const float T[16], o3r_point* out) {
    for (size_t i = 0; i < n; ++i) {
        const float x = in[i].x, y = in[i].y, z = in[i].z;
        o3r_point o;
        o.x = T[0] * x + T[1] * y + T[2] * z + T[3];
        o.y = T[4] * x + T[5] * y + T[6] * z + T[7];
        o.z = T[8] * x + T[9] * y + T[10] * z + T[11];
        o.rgb = in[i].rgb;
        out[i] = o;
    }
}

uint64_t orc_cell_key(float x, float y, float z, float lx, float ly, float lz) {
    const float ix = 1.0f / lx, iy = 1.0f / ly, iz = 1.0f / lz;
    const int64_t i = (int64_t)std::floor(x * ix), j = (int64_t)std::floor(y * iy), k = (int64_t)std::floor(z * iz);
    const int64_t B = 1 << 20;
    return ((uint64_t)(k + B) << 42) | ((uint64_t)(j + B) << 21) | (uint64_t)(i + B);
}

int orc_voxel_grid(const o3r_point* pts, size_t n, float lx, float ly, float lz, unsigned min_points,
                   o3r_point* out, size_t cap, size_t* n_out,
                   uint64_t* keys, uint32_t* counts, int* passthrough) {
    if (!n_out || (n && !pts)) return O3R_ERR_INVALID;
    if (passthrough) *passthrough = 0;
    *n_out = 0;
    if (n == 0) return O3R_OK;
    const float inv[3] = {1.0f / lx, 1.0f / ly, 1.0f / lz}; /* inverse_leaf_size_ = Ones / leaf_size_ */
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (size_t i = 0; i < n; ++i) { /* getMinMax3D */
        const float v[3] = {pts[i].x, pts[i].y, pts[i].z};
        for (int a = 0; a < 3; ++a) {
            mn[a] = std::min(mn[a], v[a]);
            mx[a] = std::max(mx[a], v[a]);
        }
    }
    /* leaf-size guard */
    const int64_t dx = (int64_t)((mx[0] - mn[0]) * inv[0]) + 1;
    const int64_t dy = (int64_t)((mx[1] - mn[1]) * inv[1]) + 1;
    const int64_t dz = (int64_t)((mx[2] - mn[2]) * inv[2]) + 1;
    if (dx * dy * dz > (int64_t)INT32_MAX) { /* "Leaf size is too small": output = input */
        if (passthrough) *passthrough = 1;
        *n_out = n;
        if (out) {
            if (cap < n) return O3R_ERR_CAPACITY;
            std::memcpy(out, pts, n * sizeof(o3r_point));
            for (size_t i = 0; i < n; ++i) {
                if (keys) keys[i] = orc_cell_key(pts[i].x, pts[i].y, pts[i].z, lx, ly, lz);
                if (counts) counts[i] = 1;
            }
        }
        return O3R_OK;
    }
    int min_b[3], max_b[3], div_b[3];
    for (int a = 0; a < 3; ++a) {
        min_b[a] = (int)std::floor(mn[a] * inv[a]);
        max_b[a] = (int)std::floor(mx[a] * inv[a]);
        div_b[a] = max_b[a] - min_b[a] + 1;
    }
    /* PCL's divb_mul_ and index are int and wrap once div_b[0]*div_b[1]*div_b[2] exceeds INT32_MAX (the guard above uses the
       slightly smaller (max - min) * inv); uint32 arithmetic gives the same bits without the undefined signed overflow */
    const uint32_t mul[3] = {1u, (uint32_t)div_b[0], (uint32_t)div_b[0] * (uint32_t)div_b[1]};
    struct IdxPt { unsigned idx; unsigned pt; };
    std::vector<IdxPt> iv(n);
    for (size_t i = 0; i < n; ++i) {
        const int i0 = (int)(std::floor(pts[i].x * inv[0]) - (float)min_b[0]);
        const int i1 = (int)(std::floor(pts[i].y * inv[1]) - (float)min_b[1]);
        const int i2 = (int)(std::floor(pts[i].z * inv[2]) - (float)min_b[2]);
        iv[i].idx = (uint32_t)i0 * mul[0] + (uint32_t)i1 * mul[1] + (uint32_t)i2 * mul[2];
        iv[i].pt = (unsigned)i;
    }
    /* PCL uses std::sort (order inside a voxel unspecified); the oracle fixes it to input order. */
    std::stable_sort(iv.begin(), iv.end(), [](const IdxPt& a, const IdxPt& b) { return a.idx < b.idx; });
    size_t total = 0;
    int rc = O3R_OK;
    for (size_t index = 0; index < n;) {
        size_t i = index + 1;
        while (i < n && iv[i].idx == iv[index].idx) ++i;
        const size_t cnt = i - index;
        if (cnt >= min_points) {
            if (out) {
                if (total < cap) {
                    /* CentroidPoint<PointXYZRGB>: AccumulatorXYZ (float sums / n), AccumulatorRGBA (float sums,
                       uint32(sum / n)) */
                    float sx = 0.f, sy = 0.f, sz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
                    for (size_t li = index; li < i; ++li) {
                        const o3r_point& q = pts[iv[li].pt];
                        sx += q.x; sy += q.y; sz += q.z;
                        sr += (float)((q.rgb >> 16) & 255u);
                        sg += (float)((q.rgb >> 8) & 255u);
                        sb += (float)(q.rgb & 255u);
                    }
                    const float fn = (float)cnt;
                    o3r_point o;
                    o.x = sx / fn; o.y = sy / fn; o.z = sz / fn;
                    o.rgb = ((uint32_t)(sr / fn) << 16) | ((uint32_t)(sg / fn) << 8) | (uint32_t)(sb / fn);
                    out[total] = o;
                    const o3r_point& q0 = pts[iv[index].pt];
                    if (keys) keys[total] = orc_cell_key(q0.x, q0.y, q0.z, lx, ly, lz);
                    if (counts) counts[total] = (uint32_t)cnt;
                } else {
                    rc = O3R_ERR_CAPACITY;
                }
            }
            ++total;
        }
        index = i;
    }
    *n_out = total;
    return rc;
}

int orc_sor(const o3r_point* pts, size_t n, int mean_k, double stddev_mul, int threads, int brute,
            uint8_t* keep, float* dist_out) {
    if ((n && !pts) || !keep || mean_k < 1) return O3R_ERR_INVALID;
    std::vector<float> dist(n);
    sor_distances(pts, n, mean_k, threads, brute != 0, dist.data());
    double sum = 0, sq_sum = 0;
    for (size_t i = 0; i < n; ++i) {
        sum += dist[i];
        sq_sum += dist[i] * dist[i];   /* float product, as in PCL */
    }
    const double mean = sum / (double)n;
    const double variance = (sq_sum - sum * sum / (double)n) / ((double)n - 1);
    const double stddev = std::sqrt(variance);
    const double threshold = mean + stddev_mul * stddev;
    for (size_t i = 0; i < n; ++i) keep[i] = !(dist[i] > threshold);
    if (dist_out) std::memcpy(dist_out, dist.data(), n * sizeof(float));
    return O3R_OK;
}

int orc_downsample_pt_cloud(const o3r_params* p, const o3r_point* pts, size_t n, int combined,
                            o3r_point* out, size_t cap, size_t* n_out) {
    std::vector<o3r_point> tmp(pts, pts + n); /* pose_functions.cpp:1660-1669 */
    if (combined)
        for (size_t i = 0; i < n; ++i) tmp[i].z += 500; /* :1666 */
    if (!combined && p->jump_pixels > 0 && p->sor_mean_k > 0) { /* :1673-1686 */
        std::vector<uint8_t> keep(n);
        int rs = orc_sor(tmp.data(), n, p->sor_mean_k, p->sor_stddev_mul, 1, 0, keep.data(), nullptr);
        if (rs) return rs;
        size_t m = 0;
        for (size_t i = 0; i < n; ++i)
            if (keep[i]) tmp[m++] = tmp[i];
        tmp.resize(m);
        n = m;
    }
    int rc;
    if (combined) { /* :1691-1695 */
        rc = orc_voxel_grid(tmp.data(), n, (float)p->voxel_size, (float)p->voxel_size, 1000.0f,
                            p->min_points_per_voxel, out, cap, n_out, nullptr, nullptr, nullptr);
        if (out) {
            const size_t m = std::min(*n_out, cap);
            for (size_t i = 0; i < m; ++i) out[i].z -= 500; /* :1702-1704 */
        }
    } else { /* :1698 */
        const float leaf = (float)(p->voxel_size / 5);
        rc = orc_voxel_grid(tmp.data(), n, leaf, leaf, leaf, 0, out, cap, n_out, nullptr, nullptr, nullptr);
    }
    return rc;
}

int orc_create_and_transform_pt_cloud(const o3r_params* p, const o3r_frame* f, int disp_type,
                                      o3r_point* out, size_t cap, size_t* n_out) {
    size_t n = 0;
    int rc = orc_create_single_img_pt_cloud(p, f, disp_type, nullptr, 0, &n, nullptr, 0, nullptr);
    if (rc) { *n_out = 0; return rc; }
    std::vector<o3r_point> cloud(n);
    rc = orc_create_single_img_pt_cloud(p, f, disp_type, cloud.data(), n, &n, nullptr, 0, nullptr);
    if (rc) { *n_out = 0; return rc; }
    orc_transform_pt_cloud(cloud.data(), n, f->T, cloud.data()); /* pose.cpp:606-607 */
    if (!p->dont_downsample) /* pose.cpp:609-613 */
        return orc_downsample_pt_cloud(p, cloud.data(), n, 0, out, cap, n_out);
    *n_out = n;
    if (out) {
        if (cap < n) return O3R_ERR_CAPACITY;
        std::memcpy(out, cloud.data(), n * sizeof(o3r_point));
    }
    return O3R_OK;
}

int orc_run_cycle(const o3r_params* p, const o3r_frame* frames, int n, int disp_type, int threads,
                  o3r_point* cloud_big, size_t cloud_cap, size_t* cloud_n, uint32_t* frame_counts) {
    if (n <= 0) return O3R_OK;
    if (threads < 1) threads = 1;
    std::vector<std::vector<o3r_point>> clouds(n);
    std::atomic<int> next(0), err(0);
    auto worker = [&]() {
        for (;;) {
            const int i = next.fetch_add(1);
            if (i >= n) break;
            /* pose.cpp:596-636: any failure inside the thread yields an empty cloud */
            size_t cap = 0, m = 0;
            if (p->jump_pixels > 0) {
                const int J = p->jump_pixels;
                const size_t nx = (size_t)((p->cols - p->bounding_box - p->cols_start_aft_cutout + J - 1) / J);
                const size_t ny = (size_t)((p->rows - 2 * p->bounding_box + J - 1) / J);
                cap = nx * ny;
            }
            if (p->jump_pixels != 1) cap += (size_t)frames[i].n_kp;
            clouds[i].resize(cap);
            int rc = orc_create_and_transform_pt_cloud(p, &frames[i], disp_type, clouds[i].data(), cap, &m);
            if (rc) { m = 0; err.store(rc); }
            clouds[i].resize(m);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(worker);
    worker();
    for (auto& t : pool) t.join();
    for (int i = 0; i < n; ++i) { /* pose.cpp:415-434 ordered concat + append */
        if (frame_counts) frame_counts[i] = (uint32_t)clouds[i].size();
        if (*cloud_n + clouds[i].size() > cloud_cap) return O3R_ERR_CAPACITY;
        std::memcpy(cloud_big + *cloud_n, clouds[i].data(), clouds[i].size() * sizeof(o3r_point));
        *cloud_n += clouds[i].size();
    }
    return O3R_OK;
}

void orc_mat4_mul(const float a[16], const float b[16], float out[16]) { mat4_mul(a, b, out); }

int orc_generate_tmat(double tx, double ty, double tz, double qx, double qy, double qz, double qw,
                      float out[16]) {
    /* pose.h:142-147 */
    const double trans_x_hi = -0.300, trans_y_hi = -0.040, trans_z_hi = -0.350;
    const double PI = 3.141592653589793238463;
    const double theta_xi = -1.1408 * PI / 180, theta_yi = 1.1945 * PI / 180;
    auto ident = [](float* m) { for (int i = 0; i < 16; ++i) m[i] = (i % 5 == 0) ? 1.0f : 0.0f; };
    auto zero = [](float* m) { for (int i = 0; i < 16; ++i) m[i] = 0.0f; };
    float r_xi[16], r_yi[16], r_invert_i[16], r_invert_y[16], t_hi[16], r_flip_xy[16], r_wh[16], t_wh[16];
    ident(r_xi); /* :1181-1190 */
    r_xi[5] = (float)std::cos(theta_xi); r_xi[6] = (float)-std::sin(theta_xi);
    r_xi[9] = (float)std::sin(theta_xi); r_xi[10] = (float)std::cos(theta_xi);
    ident(r_yi); /* :1193-1202 */
    r_yi[0] = (float)std::cos(theta_yi); r_yi[2] = (float)std::sin(theta_yi);
    r_yi[8] = (float)-std::sin(theta_yi); r_yi[10] = (float)std::cos(theta_yi);
    zero(r_invert_i); r_invert_i[15] = 1; r_invert_i[0] = 1; r_invert_i[5] = -1; r_invert_i[10] = -1; /* :1205-1213 */
    zero(r_invert_y); r_invert_y[15] = 1; r_invert_y[0] = 1; r_invert_y[5] = -1; r_invert_y[10] = 1;  /* :1214-1221 */
    ident(t_hi); t_hi[3] = (float)trans_x_hi; t_hi[7] = (float)trans_y_hi; t_hi[11] = (float)trans_z_hi; /* :1232-1240 */
    zero(r_flip_xy); r_flip_xy[15] = 1; r_flip_xy[4] = 1; r_flip_xy[1] = 1; r_flip_xy[10] = 1; /* :1243-1251 */
    const double sqw = qw * qw, sqx = qx * qx, sqy = qy * qy, sqz = qz * qz; /* :1274-1277 */
    if (sqw + sqx + sqy + sqz < 0.99 || sqw + sqx + sqy + sqz > 1.01) return -1; /* :1279-1280 */
    double rot[3][3];
    rot[0][0] = sqx - sqy - sqz + sqw; rot[1][1] = -sqx + sqy - sqz + sqw; rot[2][2] = -sqx - sqy + sqz + sqw;
    double t1 = qx * qy, t2 = qz * qw;
    rot[0][1] = 2.0 * (t1 + t2); rot[1][0] = 2.0 * (t1 - t2);
    t1 = qx * qz; t2 = qy * qw;
    rot[0][2] = 2.0 * (t1 - t2); rot[2][0] = 2.0 * (t1 + t2);
    t1 = qy * qz; t2 = qx * qw;
    rot[1][2] = 2.0 * (t1 + t2); rot[2][1] = 2.0 * (t1 - t2);
    zero(r_wh); r_wh[15] = 1; /* :1303-1311: rot = rot.t(); r_wh(i,j) = rot(i,j) */
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) r_wh[i * 4 + j] = (float)rot[j][i];
    ident(t_wh); t_wh[3] = (float)tx; t_wh[7] = (float)ty; t_wh[11] = (float)tz; /* :1317-1325 */
    float m[16]; /* :1341, evaluated left to right in float */
    mat4_mul(t_wh, r_wh, m);
    mat4_mul(m, r_invert_y, m);
    mat4_mul(m, r_flip_xy, m);
    mat4_mul(m, t_hi, m);
    mat4_mul(m, r_invert_i, m);
    mat4_mul(m, r_yi, m);
    mat4_mul(m, r_xi, m);
    std::memcpy(out, m, sizeof(m));
    return 0;
}

double orc_get_variance(const o3r_params* p, const void* img, size_t step, int plane_fitted) {
    const int rows = p->rows, cols = p->cols, bb = p->bounding_box, x0 = p->cols_start_aft_cutout;
    auto val = [&](int y, int x) -> double {
        const uint8_t* row = (const uint8_t*)img + (size_t)y * step;
        return plane_fitted ? ((const double*)row)[x] : (double)row[x];
    };
    double sum = 0.0; /* getMean :987-1005 */
    for (int y = bb; y < rows - bb; ++y)
        for (int x = x0; x < cols - bb; ++x) {
            const double d = val(y, x);
            if (d > p->min_disparity) sum += d;
        }
    const double mean = sum / ((rows - 2 * bb) * (cols - bb - x0));
    double temp = 0; /* getVariance :1007-1028 */
    for (int y = bb; y < rows - bb; ++y)
        for (int x = x0; x < cols - bb; ++x) {
            const double d = val(y, x);
            if (d > p->min_disparity) temp += (d - mean) * (d - mean);
        }
    return temp / ((rows - 2 * bb) * (cols - bb - x0) - 1);
}

int orc_plane_fit(const o3r_params* p, const uint8_t* labels, size_t labels_step,
                  const uint8_t* disp, size_t disp_step, double* coef_out, int* n_planes,
                  double* f64_out) {
    const int rows = p->rows, cols = p->cols, bb = p->bounding_box, x0 = p->cols_start_aft_cutout;
    if (f64_out) std::fill(f64_out, f64_out + (size_t)rows * cols, 0.0); /* :905 */
    int np = 0;
    for (int cluster = 1; cluster < 1024; ++cluster) { /* :907 */
        size_t total = 0;
        double sxx = 0, sxy = 0, sx = 0, syy = 0, sy = 0, s1 = 0, sxz = 0, syz = 0, sz = 0;
        for (int l = 0; l < rows; ++l)
            for (int k = 0; k < cols; ++k)
                if (labels[(size_t)l * labels_step + k] == cluster) {
                    ++total;
                    if (k > x0 && k < cols - bb && l > bb && l < rows - bb) { /* :929 strict */
                        const double X = k, Y = l, Z = (double)disp[(size_t)l * disp_step + k];
                        sxx += X * X; sxy += X * Y; sx += X; syy += Y * Y; sy += Y; s1 += 1.0;
                        sxz += X * Z; syz += Y * Z; sz += Z;
                    }
                }
        if (total == 0) break; /* :923 */
        double* c = coef_out + 3 * (cluster - 1);
        c[0] = c[1] = c[2] = 0.0;
        np = cluster;
        if (s1 == 0.0) continue; /* :939-940: label keeps 0.0 everywhere */
        /* :957-965: x = inv_SVD(AtA) * At * b */
        double A[3][3] = {{sxx, sxy, sx}, {sxy, syy, sy}, {sx, sy, s1}}, V[3][3], w[3];
        jacobi3(A, V, w);
        double wmax = std::max(std::fabs(w[0]), std::max(std::fabs(w[1]), std::fabs(w[2])));
        const double thr = DBL_EPSILON * 2 * (std::fabs(w[0]) + std::fabs(w[1]) + std::fabs(w[2]));
        (void)wmax;
        const double rhs[3] = {sxz, syz, sz};
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
        if (f64_out)
            for (int l = 0; l < rows; ++l)
                for (int k = 0; k < cols; ++k)
                    if (labels[(size_t)l * labels_step + k] == cluster) /* :968-971 */
                        f64_out[(size_t)l * cols + k] = 1.0 * c[0] * k + 1.0 * c[1] * l + 1.0 * c[2];
    }
    *n_planes = np;
    return O3R_OK;
}

/* struct sizes as the C compiler lays them out (tests compare with the ctypes mirror) */
size_t orc_sizeof(int which) {
    switch (which) {
        case 0: return sizeof(o3r_params);
        case 1: return sizeof(o3r_frame);
        case 2: return sizeof(o3r_point);
        case 3: return sizeof(o3r_cell);
        default: return 0;
    }
}

}  /* extern "C" */
