// Preprocessing of one region (SURVEY.md section 8 row f-4): per-species rescale + log transform,
// contact image, 3x3 median hole fill, Perona-Malik diffusion, node-order flatten.
// Reference: utility.py:867-897, 362, 2192-2226, 2332-2365, 603-659, 1566-1573 (medpy call),
// 2295-2329, 2368-2400.  One-shot per data set and HBM-/latency-bound; everything runs on the device
// so that a 10 kb chr1 image (6.2e8 pixels per species) never exists on the host.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace phmrf {

namespace {

constexpr double kThresh = 1e-05;  // utility.py:47 THRESH1

// ---- normalise -------------------------------------------------------------------------------
// Column minima / maxima of max(x, 0): non-negative doubles order like their bit patterns.
__global__ void colminmax_kernel(const double *__restrict__ x, int64_t n, int d, unsigned long long *mn,
                                 unsigned long long *mx) {
    const int c = blockIdx.y;
    unsigned long long lo = ~0ull, hi = 0ull;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v = x[i * d + c];
        v = v < 0 ? 0.0 : v;  // (a NaN stays a NaN and is not ordered: left to the caller like numpy's min)
        const unsigned long long b = (unsigned long long)__double_as_longlong(v + 0.0);
        lo = b < lo ? b : lo;
        hi = b > hi ? b : hi;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(mn + c, lo);
        atomicMax(mx + c, hi);
    }
}

// x = x_min + (x - m1) * 1.0 * (x_max - x_min) / (m2 - m1), then log(1 + x); numpy's operation
// order, no contraction.
__global__ void rescale_kernel(double *__restrict__ x, int64_t n, int d, const double *__restrict__ colmm, double x_min,
                               double x_max, int log1p) {
    const double span = __dsub_rn(x_max, x_min);
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n * d; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % d);
        const double m1 = colmm[2 * c], m2 = colmm[2 * c + 1];
        double v = x[e];
        v = v < 0 ? 0.0 : v;
        double y = __dmul_rn(__dmul_rn(__dsub_rn(v, m1), 1.0), span);
        y = __ddiv_rn(y, __dsub_rn(m2, m1));
        y = __dadd_rn(x_min, y);
        x[e] = log1p ? log(__dadd_rn(1.0, y)) : y;
    }
}

// ---- image -----------------------------------------------------------------------------------
__global__ void scatter_kernel(const double *__restrict__ value, const int64_t *__restrict__ pos, int64_t n, int d,
                               int c, int64_t start1, int64_t start2, int64_t n1, int64_t n2, int symmetric,
                               double *__restrict__ plane, int *bad) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t a = pos[2 * i] - start1, b = pos[2 * i + 1] - start2;
        if (a < 0 || b < 0 || a >= n1 || b >= n2 || (symmetric && (b >= n1 || a >= n2))) {
            *bad = 1;
            continue;
        }
        const double v = value[i * d + c];
        plane[a * n2 + b] = v;
        if (symmetric) plane[b * n2 + a] = v;
    }
}

// median of the 8 neighbours = mean of the 4th and 5th smallest (numpy.median of an even count).
// A 17-comparator selection network of depth 6 (the 19-comparator sorting network for 8 keys with the two
// exchanges that cannot reach outputs 3 and 4 removed; checked exhaustively with the 0-1 principle): the
// hole fill is a chain of dependent steps, so the DEPTH of the network is what its run time is made of.
__device__ __forceinline__ void cmpx(double &a, double &b) {
    const double lo = fmin(a, b), hi = fmax(a, b);
    a = lo;
    b = hi;
}
__device__ __forceinline__ double median8(double (&w)[8]) {
    cmpx(w[0], w[1]); cmpx(w[2], w[3]); cmpx(w[4], w[5]); cmpx(w[6], w[7]);
    cmpx(w[0], w[2]); cmpx(w[1], w[3]); cmpx(w[4], w[6]); cmpx(w[5], w[7]);
    cmpx(w[1], w[2]); cmpx(w[5], w[6]); cmpx(w[0], w[4]); cmpx(w[3], w[7]);
    cmpx(w[1], w[5]); cmpx(w[2], w[6]);
    cmpx(w[2], w[4]); cmpx(w[3], w[5]);
    cmpx(w[3], w[4]);
    return __dmul_rn(__dadd_rn(w[3], w[4]), 0.5);  // = (a+b)/2 correctly rounded, without the division routine
}

// 3x3 median hole fill in the reference's sequential raster order (utility.py:603-659).  Cell (i,j)
// reads row i-1 and (i,j-1) -- already updated -- and (i,j+1), row i+1 -- not yet updated.  In the
// skewed coordinates (i, s = i + j) every updated neighbour has a smaller or equal i AND a smaller or
// equal s, and every not-yet-updated one a larger or equal i and s; so the (i, s) plane can be cut
// into rectangular tiles (kHfR rows x kHfC skewed columns), a tile depends only on its upper, left
// and upper-left neighbours, and all tiles with the same I + S are independent: one launch per tile
// anti-diagonal, one warp per tile.  Inside a tile the cells with equal ri + si (= the 2i + j fronts
// of the unskewed image) are independent as well: lane = row, kHfR + kHfC - 1 steps with a warp
// barrier, on a shared-memory copy of the tile's bounding box (row stride odd: conflict free).  The
// result equals the sequential scan bit for bit (the CPU test tier replays this schedule on
// the CPU; tests/test_gpu_prep.py compares with the reference's fixtures).
// symmetric != 0: only the upper triangle (j >= i) is scanned and a cell below the diagonal is read
// through its mirror, which is what the reference's mirrored writes amount to on a symmetric image;
// the lower triangle is rewritten afterwards (mirror_kernel).
// (Round 1 swept the 2i+j fronts of the WHOLE image with one CTA per plane: 3W block barriers and one
// 32-byte sector per cell, 117 ms at W = 8192.)
constexpr int kHfR = 32, kHfC = 64;
constexpr int kHfBH = kHfR + 2, kHfBW = kHfC + kHfR + 1;  // bounding box incl. the one-cell halo; width odd
constexpr int kHfThreads = 128;  // four warps fetch the bounding box (the loads are the latency), warp 0 sweeps the tile

__global__ void __launch_bounds__(kHfThreads) holefill_tile_kernel(double *__restrict__ planes, int64_t plane_stride, int64_t n1,
                                                           int64_t n2, int symmetric, int w, int I_lo) {
    __shared__ double tile[kHfBH][kHfBW];
    const int I = I_lo + (int)blockIdx.x, S = w - I;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *P = planes + (int64_t)blockIdx.y * plane_stride;
    const int64_t i0 = (int64_t)I * kHfR, s0 = (int64_t)S * kHfC;
    const int64_t i_lo = 2, i_hi = n1 - 2, j_hi = n2 - 2;  // inclusive bounds of range(2, n-1)
    // does the tile hold any cell of the scan?  rows [i0, i0+R) x columns j = s - i
    const int64_t ra = i0 > i_lo ? i0 : i_lo, rb = (i0 + kHfR - 1) < i_hi ? (i0 + kHfR - 1) : i_hi;
    if (ra > rb) return;
    if (s0 + kHfC - 1 - ra < (symmetric ? ra : 2)) return;  // largest j of the tile (at its first scanned row)
    if (s0 - rb > j_hi) return;                             // smallest j of the tile (at its last scanned row)
    const int64_t bi0 = i0 - 1, bj0 = s0 - (i0 + kHfR - 1) - 1;
    constexpr int kCols = (kHfBW + 31) / 32;
#pragma unroll 3
    for (int r = warp; r < kHfBH; r += kHfThreads / 32) {
        const int64_t gi = bi0 + r;
        double v[kCols];
#pragma unroll
        for (int q = 0; q < kCols; ++q) {  // all loads of a row in flight before the first store
            const int c = lane + 32 * q;
            const int64_t gj = bj0 + c;
            v[q] = (c < kHfBW && gi >= 0 && gi < n1 && gj >= 0 && gj < n2) ? P[gi * n2 + gj] : 0.0;
        }
#pragma unroll
        for (int q = 0; q < kCols; ++q)
            if (lane + 32 * q < kHfBW) tile[r][lane + 32 * q] = v[q];
    }
    __syncthreads();
    if (warp != 0) return;
    // lane = row; at step d the lane's cell sits at bounding-box column c = d - 2*lane + kHfR (one column further
    // per step).  Everything that does not change along the row is worked out once: the columns of the row that
    // belong to this tile AND to the scan, the column up to which a neighbour may lie below the diagonal (read
    // through its mirror), the row's address in the plane.
    const int64_t i = i0 + lane;
    const bool row_ok = i >= i_lo && i <= i_hi;
    const int64_t j_first = symmetric ? i : 2;
    int c_min = kHfR - lane, c_max = kHfR - lane + kHfC - 1;                 // the tile's own skewed columns
    if (j_first - bj0 > c_min) c_min = (int)(j_first - bj0);                  // the scan's range of j
    if (j_hi - bj0 < c_max) c_max = (int)(j_hi - bj0);
    if (!row_ok) c_max = c_min - 1;
    const int c_diag = symmetric ? (int)(i + 1 - bj0) : -1;                   // j <= i + 1: a neighbour has a > b
    double *const Prow = P + i * n2 + bj0;
    double *const trow = &tile[lane + 1][0];
    int c = kHfR - 2 * lane;
    for (int d = 0; d < kHfR + kHfC - 1; ++d, ++c) {
        if (c >= c_min && c <= c_max && trow[c] < kThresh) {
            double nb[8];
            if (c > c_diag) {                       // all eight neighbours on or above the diagonal: fixed offsets
                const double *q = trow + c;
                nb[0] = q[-kHfBW - 1]; nb[1] = q[-kHfBW]; nb[2] = q[-kHfBW + 1];
                nb[3] = q[-1];                            nb[4] = q[1];
                nb[5] = q[kHfBW - 1];  nb[6] = q[kHfBW];  nb[7] = q[kHfBW + 1];
            } else {
                const int64_t j = c + bj0;
                int q = 0;
#pragma unroll
                for (int di = -1; di <= 1; ++di)
#pragma unroll
                    for (int dj = -1; dj <= 1; ++dj) {
                        if (di == 0 && dj == 0) continue;
                        int64_t a = i + di, b = j + dj;
                        if (a > b) {
                            const int64_t t = a;
                            a = b;
                            b = t;
                        }
                        nb[q++] = tile[(int)(a - bi0)][(int)(b - bj0)];
                    }
            }
            const double m1 = median8(nb);
            if (m1 > kThresh) {
                trow[c] = m1;
                Prow[c] = m1;
            }
        }
        __syncwarp();
    }
}

// every tile anti-diagonal in turn (stream order is the only synchronisation between them)
static int launch_holefill(double *planes, int64_t plane_stride, int nb, int64_t n1, int64_t n2, int symmetric,
                           cudaStream_t s) {
    if (n1 - 2 < 2 || n2 - 2 < 2) return PHMRF_OK;
    const int NI = (int)((n1 + kHfR - 1) / kHfR), NS = (int)((n1 + n2 - 1 + kHfC - 1) / kHfC);
    for (int w = 0; w < NI + NS - 1; ++w) {
        const int I_lo = w - NS + 1 > 0 ? w - NS + 1 : 0, I_hi = w < NI - 1 ? w : NI - 1;
        holefill_tile_kernel<<<dim3(I_hi - I_lo + 1, nb), kHfThreads, 0, s>>>(planes, plane_stride, n1, n2, symmetric, w, I_lo);
    }
    count_launch(NI + NS - 1);
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

__global__ void mirror_kernel(double *__restrict__ P, int64_t n) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n * n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = e / n, j = e % n;
        if (i > j) P[e] = P[j * n + i];
    }
}

__global__ void to_f32_kernel(const double *__restrict__ in, float *__restrict__ out, int64_t count) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
        out[e] = __double2float_rn(in[e]);
}
__global__ void to_f64_kernel(const float *__restrict__ in, double *__restrict__ out, int64_t count) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
        out[e] = (double)in[e];
}

// flux through the forward difference delta: exp(-(delta/kappa)^2) / 1 * delta, float32, numpy order
__device__ __forceinline__ float pm_flux(float delta, float kappa) {
    const float q = __fdiv_rn(delta, kappa);
    return __fmul_rn(expf(-__fmul_rn(q, q)), delta);
}

// One Perona-Malik step (medpy option 1): forward differences that vanish on the last row/column,
// flux divergence by backward differences (the first row/column keeps its own flux), out = in +
// gamma * (NS + EW).  4 B read + 4 B written per pixel (neighbours come from L1/L2).
__global__ void __launch_bounds__(256) diffuse_kernel(const float *__restrict__ in, float *__restrict__ out, int64_t n1,
                                                      int64_t n2, float kappa, float gamma) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= n2) return;
    for (int64_t i = blockIdx.y; i < n1; i += gridDim.y) {
        const float c = in[i * n2 + j];
        const float fs = i + 1 < n1 ? pm_flux(__fsub_rn(in[(i + 1) * n2 + j], c), kappa) : 0.0f;
        const float fe = j + 1 < n2 ? pm_flux(__fsub_rn(in[i * n2 + j + 1], c), kappa) : 0.0f;
        const float ns = i > 0 ? __fsub_rn(fs, pm_flux(__fsub_rn(c, in[(i - 1) * n2 + j]), kappa)) : fs;
        const float ew = j > 0 ? __fsub_rn(fe, pm_flux(__fsub_rn(c, in[i * n2 + j - 1]), kappa)) : fe;
        out[i * n2 + j] = __fadd_rn(c, __fmul_rn(gamma, __fadd_rn(ns, ew)));
    }
}

// One axis of scipy.ndimage.gaussian_filter (order 0, mode 'reflect'): symmetric correlation in
// scipy's summation order (NI_Correlate1D: centre tap first, then the pairs from the outermost in),
// separate multiply and add.
__global__ void __launch_bounds__(256) gauss1d_kernel(const double *__restrict__ in, double *__restrict__ out, int64_t n1,
                                                      int64_t n2, int axis, const double *__restrict__ w, int lw) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= n2) return;
    const int64_t len = axis == 0 ? n1 : n2, stride = axis == 0 ? n2 : 1;
    for (int64_t i = blockIdx.y; i < n1; i += gridDim.y) {
        const int64_t pos = axis == 0 ? i : j;
        const double *line = in + (axis == 0 ? j : i * n2);
        auto at = [&](int64_t k) {  // 'reflect': d c b a | a b c d | d c b a
            const int64_t per = 2 * len;
            k %= per;
            if (k < 0) k += per;
            if (k >= len) k = per - 1 - k;
            return line[k * stride];
        };
        double tmp = __dmul_rn(at(pos), w[lw]);
        for (int jj = -lw; jj < 0; ++jj)
            tmp = __dadd_rn(tmp, __dmul_rn(__dadd_rn(at(pos + jj), at(pos - jj)), w[jj + lw]));
        out[i * n2 + j] = tmp;
    }
}

// node order: upper triangle row by row (kind 1) or the whole block (kind 0)
__global__ void flatten_kernel(const double *__restrict__ plane, int64_t n1, int64_t n2, int kind, int d, int c,
                               double *__restrict__ data) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    for (int64_t i = blockIdx.y; i < n1; i += gridDim.y) {
        if (kind == 1) {
            if (j < i || j >= n2) continue;
            const int64_t row_start = i * n2 - i * (i - 1) / 2;  // nodes before row i
            data[(row_start + (j - i)) * d + c] = plane[i * n2 + j];
        } else {
            if (j >= n2) continue;
            data[(i * n2 + j) * d + c] = plane[i * n2 + j];
        }
    }
}

__global__ void interleave_kernel(const double *__restrict__ plane, int64_t count, int d, int c, double *__restrict__ img) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
        img[e * d + c] = plane[e];
}

inline int grid_for(int64_t count, int cap = 148 * 16) {
    const int64_t b = (count + 255) / 256;
    return (int)(b < 1 ? 1 : (b < cap ? b : cap));
}

}  // namespace

}  // namespace phmrf

using namespace phmrf;

extern "C" int phmrf_prep_normalise(int device, double *x, int64_t n, int d, double *x_min, double *x_max,
                                    double *colminmax_out, int log1p) {
    if (!x || n <= 0 || d <= 0 || !x_min || !x_max) {
        set_error("phmrf_prep_normalise: bad argument");
        return PHMRF_E_INVALID;
    }
    PHMRF_CUDA(cudaSetDevice(device));
    DevBuf<double> dx, dmm;
    DevBuf<unsigned long long> dmn, dmx;
    int rc;
    if ((rc = dx.alloc(n * d)) || (rc = dmn.alloc(d)) || (rc = dmx.alloc(d)) || (rc = dmm.alloc(2 * d))) return rc;
    PHMRF_CUDA(cudaMemcpy(dx, x, sizeof(double) * n * d, cudaMemcpyHostToDevice));
    PHMRF_CUDA(cudaMemset(dmn, 0xff, sizeof(unsigned long long) * d));
    PHMRF_CUDA(cudaMemset(dmx, 0, sizeof(unsigned long long) * d));
    dim3 g1((unsigned)grid_for(n, 148 * 4), (unsigned)d);
    colminmax_kernel<<<g1, 256>>>(dx, n, d, dmn, dmx);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    std::vector<unsigned long long> hmn(d), hmx(d);
    PHMRF_CUDA(cudaMemcpy(hmn.data(), dmn, sizeof(unsigned long long) * d, cudaMemcpyDeviceToHost));
    PHMRF_CUDA(cudaMemcpy(hmx.data(), dmx, sizeof(unsigned long long) * d, cudaMemcpyDeviceToHost));
    std::vector<double> mm(2 * (size_t)d), lo(d), hi(d);
    for (int c = 0; c < d; ++c) {
        memcpy(&mm[2 * c], &hmn[c], 8);
        memcpy(&mm[2 * c + 1], &hmx[c], 8);
        lo[c] = mm[2 * c];
        hi[c] = mm[2 * c + 1];
    }
    auto median = [](std::vector<double> v) {  // numpy.median: mean of the two middle values
        std::sort(v.begin(), v.end());
        const size_t m = v.size();
        return (m & 1) ? v[m / 2] : (v[m / 2 - 1] + v[m / 2]) / 2.0;
    };
    if (*x_min < 0) *x_min = median(lo);
    if (*x_max < 0) *x_max = median(hi);
    if (colminmax_out) memcpy(colminmax_out, mm.data(), sizeof(double) * 2 * d);
    PHMRF_CUDA(cudaMemcpy(dmm, mm.data(), sizeof(double) * 2 * d, cudaMemcpyHostToDevice));
    rescale_kernel<<<grid_for(n * d), 256>>>(dx, n, d, dmm, *x_min, *x_max, log1p);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    PHMRF_CUDA(cudaMemcpy(x, dx, sizeof(double) * n * d, cudaMemcpyDeviceToHost));
    return PHMRF_OK;
}

extern "C" int phmrf_prep_region_image(int device, const double *value, const int64_t *pos, int64_t n, int d, int kind,
                                       int64_t start1, int64_t start2, int64_t n1, int64_t n2, int filter_mode,
                                       int niter, double kappa, double gamma, double sigma, double *data_out,
                                       double *image_out) {
    if (!value || !pos || n <= 0 || d <= 0 || n1 <= 0 || n2 <= 0 || !data_out || (kind != 0 && kind != 1) ||
        (kind == 1 && (n1 != n2 || start1 != start2))) {
        set_error("phmrf_prep_region_image: bad argument");
        return PHMRF_E_INVALID;
    }
    PHMRF_CUDA(cudaSetDevice(device));
    const int64_t npix = n1 * n2;
    const int64_t n_nodes = kind == 1 ? n1 * (n1 + 1) / 2 : npix;
    DevBuf<double> dval, dplane, ddata, dimg, dgw, dtmp;
    DevBuf<int64_t> dpos;
    DevBuf<float> df0, df1;
    DevBuf<int> dbad;
    int lw = 0, rc;
    if (filter_mode == 2 && sigma > 0) {
        // scipy.ndimage._filters._gaussian_kernel1d: radius int(4 sigma + 0.5), exp(-x^2 / (2 sigma^2)) normalised
        lw = (int)(4.0 * sigma + 0.5);
        std::vector<double> gw(2 * (size_t)lw + 1);
        const double s2 = sigma * sigma;
        double tot = 0.0;
        for (int x = -lw; x <= lw; ++x) {
            gw[x + lw] = std::exp(-0.5 / s2 * ((double)x * (double)x));
            tot += gw[x + lw];
        }
        for (auto &v : gw) v /= tot;
        if ((rc = dgw.alloc((int64_t)gw.size())) || (rc = dtmp.alloc(npix))) return rc;
        PHMRF_CUDA(cudaMemcpy(dgw, gw.data(), sizeof(double) * gw.size(), cudaMemcpyHostToDevice));
    }
    // species are independent: the (latency-bound, one CTA per plane) hole fill runs for a batch of
    // planes at once, as many as fit a 48 GB budget
    int batch = (int)std::max<int64_t>(1, std::min<int64_t>(d, (int64_t)48e9 / (int64_t)(sizeof(double) * npix)));
    if ((rc = dval.alloc(n * d)) || (rc = dpos.alloc(2 * n)) || (rc = dplane.alloc(npix * batch)) ||
        (rc = ddata.alloc(n_nodes * d)) || (rc = dbad.alloc(1)))
        return rc;
    if (filter_mode == 0 && niter > 0 && ((rc = df0.alloc(npix)) || (rc = df1.alloc(npix)))) return rc;
    if (image_out && (rc = dimg.alloc(npix * d))) return rc;
    PHMRF_CUDA(cudaMemcpy(dval, value, sizeof(double) * n * d, cudaMemcpyHostToDevice));
    PHMRF_CUDA(cudaMemcpy(dpos, pos, sizeof(int64_t) * 2 * n, cudaMemcpyHostToDevice));
    PHMRF_CUDA(cudaMemset(dbad, 0, sizeof(int)));
    const dim3 g2((unsigned)((n2 + 255) / 256), (unsigned)(n1 < 4096 ? n1 : 4096));
    for (int c0 = 0; c0 < d; c0 += batch) {
        const int nb = std::min(batch, d - c0);
        PHMRF_CUDA(cudaMemsetAsync(dplane, 0, sizeof(double) * npix * nb));
        for (int q = 0; q < nb; ++q)
            scatter_kernel<<<grid_for(n), 256>>>(dval, dpos, n, d, c0 + q, start1, start2, n1, n2, kind == 1,
                                                 dplane + (int64_t)q * npix, dbad);
        count_launch(nb);
        {
            const int rc_fill = launch_holefill(dplane, npix, nb, n1, n2, kind == 1, nullptr);
            if (rc_fill != PHMRF_OK) return rc_fill;
        }
        for (int q = 0; q < nb; ++q) {
            const int c = c0 + q;
            double *plane = dplane + (int64_t)q * npix;
            if (kind == 1) {
                mirror_kernel<<<grid_for(npix), 256>>>(plane, n1);
                count_launch();
            }
            if (filter_mode == 0 && niter > 0) {
                float *a = df0, *b = df1;
                to_f32_kernel<<<grid_for(npix), 256>>>(plane, a, npix);
                for (int it = 0; it < niter; ++it) {
                    diffuse_kernel<<<g2, 256>>>(a, b, n1, n2, (float)kappa, (float)gamma);
                    std::swap(a, b);
                }
                to_f64_kernel<<<grid_for(npix), 256>>>(a, plane, npix);
                count_launch(niter + 2);
            }
            if (filter_mode == 2 && sigma > 0) {  // axis 0 then axis 1, like scipy
                gauss1d_kernel<<<g2, 256>>>(plane, dtmp, n1, n2, 0, dgw, lw);
                gauss1d_kernel<<<g2, 256>>>(dtmp, plane, n1, n2, 1, dgw, lw);
                count_launch(2);
            }
            flatten_kernel<<<g2, 256>>>(plane, n1, n2, kind, d, c, ddata);
            count_launch();
            if (image_out) {
                interleave_kernel<<<grid_for(npix), 256>>>(plane, npix, d, c, dimg);
                count_launch();
            }
        }
        PHMRF_CUDA(cudaGetLastError());
    }
    int bad = 0;
    PHMRF_CUDA(cudaMemcpy(&bad, dbad, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) {
        set_error("phmrf_prep_region_image: a bin pair lies outside the region window");
        return PHMRF_E_INVALID;
    }
    PHMRF_CUDA(cudaMemcpy(data_out, ddata, sizeof(double) * n_nodes * d, cudaMemcpyDeviceToHost));
    if (image_out) PHMRF_CUDA(cudaMemcpy(image_out, dimg, sizeof(double) * npix * d, cudaMemcpyDeviceToHost));
    return PHMRF_OK;
}
