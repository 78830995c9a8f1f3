// Pieces shared by the two phase-B kernels (kernels_b.cu: general path; estep_bulk.cuh:
// warp-specialised pipeline): register-tile geometry, compile-time feature rows, exp().
#pragma once
#include <cfloat>
#include <utility>

#include "common.cuh"

namespace phmrf {
namespace estep {

constexpr int kThreads = 256;
constexpr int kFastSlots = 8;  // neighbour slots kept in registers by the fast node phase

__host__ __device__ constexpr int even_up(int v) { return (v + 1) & ~1; }
// row strides (in doubles) are even (16-byte alignment of every row) with stride/2 odd, so
// that the 128-bit column accesses of the node phase are bank-conflict free.
__host__ __device__ constexpr int pad_row(int v) { return (even_up(v) / 2) % 2 == 1 ? even_up(v) : even_up(v) + 2; }

// Stride (in doubles) between the register tiles of one row: the stat phase reads `ntiles`
// different 16-byte chunks of a row in one LDS.128, which is conflict free when the chunk
// starts are at least 4 banks apart modulo 32.
__host__ __device__ constexpr bool stride_ok(int S, int ntiles) {
    for (int t1 = 0; t1 < ntiles; ++t1)
        for (int t2 = t1 + 1; t2 < ntiles; ++t2) {
            const int dd = ((t2 - t1) * S * 2) % 32;
            if (dd < 4 || dd > 28) return false;
        }
    return true;
}
__host__ __device__ constexpr int tile_stride(int T, int ntiles) {
    for (int S = even_up(T); S <= even_up(T) + 16; S += 2)
        if (stride_ok(S, ntiles)) return S;
    return even_up(T);
}

// N independent exponentials evaluated in lock step (explicit instruction-level
// parallelism for warps that cannot rely on occupancy): same reduction as exp_sm, degree-9
// polynomial (7e-12 relative, two orders below the 1e-9 parity tolerance).  CHECK=false assumes 0 <= t < 700 (results are normal numbers); CHECK=true
// additionally flushes results below 2^-1021 -- and any argument the magic-constant
// reduction cannot represent, i.e. t <= -2^27 -- to zero; arguments must not exceed +700.
// CHECK=2 instead clamps the argument from below at about -704 with one integer instruction
// (unsigned minimum on the high word): results that would be below exp(-705) ~ 7e-307 come
// out as a number in [exp(-705), exp(-704)] rather than 0 -- for soft-max terms whose sum is
// at least 1 that is an absolute error below 1e-306.
template <int N, int CHECK>
__device__ __forceinline__ void exp_batch(double (&t)[N]) {
    const double kMagic = 6755399441055744.0;
    double sft[N], r[N], p[N];
    if (CHECK == 2) {
#pragma unroll
        for (int u = 0; u < N; ++u)
            t[u] = __hiloint2double((int)min((unsigned)__double2hiint(t[u]), 0xC0860000u), __double2loint(t[u]));
    }
#pragma unroll
    for (int u = 0; u < N; ++u) sft[u] = fma(t[u], 1.4426950408889634, kMagic);
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const double fn = sft[u] - kMagic;
        r[u] = fma(fn, -6.93147180559945286e-01, t[u]);
        r[u] = fma(fn, -2.31904681384629956e-17, r[u]);
    }
    // degree-9 Taylor polynomial on |r| <= ln2/2: truncation error < 7e-12 relative
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(2.75573192239858907e-06, r[u], 2.48015873015873016e-05);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 1.98412698412698413e-04);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 1.38888888888888894e-03);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 8.33333333333333322e-03);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 4.16666666666666644e-02);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 1.66666666666666657e-01);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 0.5);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 1.0);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], r[u], 1.0);
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int n = __double2loint(sft[u]);
        int hi = __double2hiint(p[u]) + n * 1048576;
        int lo = __double2loint(p[u]);
        if (CHECK == 1) {
            // the reduction is valid while sft stays within 2^31 of the magic constant
            const bool valid = (unsigned)(__double2hiint(sft[u]) - 0x4337ffff) <= 1u;
            const bool zero = !valid || n < -1021;
            hi = zero ? 0 : hi;
            lo = zero ? 0 : lo;
        }
        t[u] = __hiloint2double(hi, lo);
    }
}

template <int D, int TK, int TF>
struct Cfg {
    static constexpr int F = n_stat_features(D);
    static constexpr int NFT = (F + TF - 1) / TF;
    static constexpr int NKT_MAX = 32 / NFT;
    static constexpr int TKs = tile_stride(TK, NKT_MAX);
    static constexpr int TFs = tile_stride(TF, NFT);
    static constexpr int RSY = pad_row(NFT * TFs);
};

// ---- per-node feature row, resolved at compile time ------------------------------------
__host__ __device__ constexpr int tri_row_of(int r, int D) {
    int i = 0;
    while (r >= D - i) {
        r -= D - i;
        ++i;
    }
    return i;
}
__host__ __device__ constexpr int tri_col_of(int r, int D) {
    int i = 0;
    while (r >= D - i) {
        r -= D - i;
        ++i;
    }
    return i + r;
}

// value stored at position POS of the Y row: feature f = tile*TF + off, or 0 on padding.
template <int D, int TF, int TFs, int POS>
__device__ __forceinline__ double y_at(const double (&x)[D], const double (&xs)[D], double inv) {
    constexpr int F = n_stat_features(D);
    constexpr int NFT = (F + TF - 1) / TF;
    constexpr int tile = POS / TFs, off = POS % TFs;
    constexpr int f = tile * TF + off;
    if constexpr (tile >= NFT || off >= TF || f >= F) {
        return 0.0;
    } else if constexpr (f == 0) {
        return inv;
    } else if constexpr (f <= D) {
        return xs[f - 1];
    } else {
        constexpr int r = f - 1 - D;
        return xs[tri_row_of(r, D)] * x[tri_col_of(r, D)];
    }
}

template <int D, int TF, int TFs, int... Cs>
__device__ __forceinline__ void write_y_row(double *Yrow, const double (&x)[D], const double (&xs)[D], double inv,
                                            std::integer_sequence<int, Cs...>) {
    ((*reinterpret_cast<double2 *>(Yrow + 2 * Cs) =
          make_double2(y_at<D, TF, TFs, 2 * Cs>(x, xs, inv), y_at<D, TF, TFs, 2 * Cs + 1>(x, xs, inv))),
     ...);
}

// 1/a for a normal, positive a: hardware seed + two Newton steps (full double precision up to
// an ulp or two; no IEEE rounding or special-case branches like the `/` operator).
__device__ __forceinline__ double fast_rcp(double a) {
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(a));
    double e = fma(-a, x, 1.0);
    x = fma(x, e, x);
    e = fma(-a, x, 1.0);
    return fma(x, e, x);
}

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// exp() for the soft-max terms: round-to-nearest range reduction with the 2^52+2^51 magic
// constant, two-term ln2, degree-11 polynomial on |r| <= ln2/2 (truncation error < 7e-15
// relative), exponent patched in with integer adds.  Results below 2^-1021 flush to 0,
// arguments beyond the double range (and NaN) return +inf, which the callers treat as
// "redo on the exact path"; no branches, ~15 FP64-pipe instructions
// (libdevice exp() measured ~50 instructions per call here, mostly range handling).
__device__ __forceinline__ double exp_sm(double t) {
    const double kMagic = 6755399441055744.0;
    const double s = fma(t, 1.4426950408889634, kMagic);
    const int n = __double2loint(s);
    const double fn = s - kMagic;
    double r = fma(fn, -6.93147180559945286e-01, t);
    r = fma(fn, -2.31904681384629956e-17, r);
    double p = 2.50521083854417188e-08;               // 1/11!
    p = fma(p, r, 2.75573192239858907e-07);           // 1/10!
    p = fma(p, r, 2.75573192239858907e-06);           // 1/9!
    p = fma(p, r, 2.48015873015873016e-05);           // 1/8!
    p = fma(p, r, 1.98412698412698413e-04);           // 1/7!
    p = fma(p, r, 1.38888888888888894e-03);           // 1/6!
    p = fma(p, r, 8.33333333333333322e-03);           // 1/5!
    p = fma(p, r, 4.16666666666666644e-02);           // 1/4!
    p = fma(p, r, 1.66666666666666657e-01);           // 1/3!
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    int hi = __double2hiint(p) + n * 1048576;
    int lo = __double2loint(p);
    // |t| >= 2^27 (incl. +-inf): the magic-constant reduction no longer holds; decide by sign
    const int thi = __double2hiint(t);
    const bool huge = (thi & 0x7ff00000) >= 0x41a00000;
    const bool under = n < -1021 || (huge && thi < 0);
    const bool over = (n > 1023 && !huge) || (huge && thi >= 0);
    hi = under ? 0 : (over ? 0x7ff00000 : hi);
    lo = (under || over) ? 0 : lo;
    return __hiloint2double(hi, lo);
}

struct TileChoice {
    int tk, tf;
};

// One (TK,TF) register tile per feature count; TF*NFT >= F with little waste, TK*TF <= 60.
constexpr TileChoice tile_for(int D) {
    switch (D) {
        case 1: return {8, 3};
        case 2: return {8, 6};
        case 3: return {5, 10};
        case 4: return {6, 8};
        case 5: return {5, 11};
        case 6: return {4, 14};
        case 7: return {5, 12};
        case 8: return {4, 15};
        case 9: return {5, 11};
        case 10: return {5, 11};
        case 11: return {4, 13};
        default: return {4, 13};
    }
}


}  // namespace estep
}  // namespace phmrf
