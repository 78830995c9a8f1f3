// Phase B, bulk-copy pipeline (the fast path for the reference's own model shape: Potts
// compatibility, <= 8 neighbour slots, K <= 40 states).  Same arithmetic as kernels_b.cu
// (reference: phylo_hmrf.py:311-314, 334-468).
//
// One CTA per SM, 4 + P warps (P = 12 where shared memory allows, else 8 or 4):
//   warps 0-3   CONSUMERS (one per SM sub-partition): hold the K x F sufficient-statistic
//               accumulators and issue nothing but  S[k][f] += e[n][k] * y[n][f]  as DMMA.8x8x4
//               (mma.sync m8n8k4 f64; on B200 it shares the DFMA datapath, but one instruction
//               carries 256 FMAs and takes one operand per lane).
//   warps 4..   PRODUCERS: the per-node work for tiles of 32 nodes, one lane per node;
//               producer p feeds consumer p % 4.
// Shared memory, every buffer [row][32 nodes]:
//   E buffer, one per producer [KP rows]   the log-likelihood tile, fetched by ONE cp.async.bulk
//               (the HBM layout is tile-major and pre-swizzled, common.cuh lp_index) onto an
//               mbarrier; the soft-max terms e_k = exp(logp_k - shift) * G_k are formed in place,
//               8 states at a time, so no per-state register row exists.  Before the copy is
//               issued the same buffer serves as scratch for the neighbour products
//               G_k = exp(sum of beta*w over the neighbours labelled k), built multiplicatively
//               slot by slot and read back as one factor per neighbour slot.
//   Y slots, two per consumer [FP rows]    the feature rows y_f / sum(e), y = (1, x, x (x) x
//               packed), written once the normaliser is known; claimed in tile order.
// Every row is XOR-swizzled by (row % 8) * 4 columns: lane-per-node accesses along a row and
// the mma operand fragments (8 rows x 4 nodes) are both bank-conflict free
// (tools/swizzle_check.py), and a consumer addresses every operand of a step from
// base ^ (step << 5) plus an immediate per 8-row tile.
// exp() is a 2048-entry table (2^(j/2048), shared memory) times a quadratic: 6 FP64 instructions.
// The variants measured and rejected for this kernel (neighbour data one tile ahead, sixteen producers, other
// register budgets) are recorded in profiles/r2_history.md.
#pragma once
#include "estep_common.cuh"

namespace phmrf {

using namespace estep;

namespace {

constexpr int kCons = 4;
constexpr int kTile = 32;
constexpr int kExpTab = 2048;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.u32 %0, 1, 0, p; }"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
// one contiguous run global -> shared through the bulk-copy engine, completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// D(8x8) += A(8x4) * B(4x8), FP64.  Lane (g = lane/4, t = lane%4) supplies A[g][t], B[t][g]
// and holds D[g][2t], D[g][2t+1].
__device__ __forceinline__ void dmma_8x8x4(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// N independent exponentials in lock step: t = (n + j/2048) ln2 + r, |r| <= ln2/4096,
// exp(t) = 2^n * tab[j] * (1 + r + r^2/2)   (truncation r^3/6 < 9e-13 relative; the one-constant
// reduction r = t - fn*(ln2/2048) is exact in the product and off by fn * 2.7e-20 < 6e-14).
// The argument is clamped from below at about -704 with one integer minimum on the high word
// (results that would be below exp(-705) come out in [exp(-705), exp(-704)] instead of 0: for
// soft-max terms whose sum is at least 1 an absolute error below 1e-306); it must not exceed
// +700.  6 FP64-pipe instructions per value (the Taylor form of round 1 took 13): every FP64
// instruction of a per-node warp competes with the DMMA stream of its sub-partition.
template <int N>
__device__ __forceinline__ void exp_tab(double (&t)[N], const double *tab) {
    const double kMagic = 6755399441055744.0;
    double sft[N], p[N];
#pragma unroll
    for (int u = 0; u < N; ++u)
        t[u] = __hiloint2double((int)min((unsigned)__double2hiint(t[u]), 0xC0860000u), __double2loint(t[u]));
#pragma unroll
    for (int u = 0; u < N; ++u) sft[u] = fma(t[u], 2954.639443740597, kMagic);
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const double fn = sft[u] - kMagic;
        t[u] = fma(fn, -0x1.62e42fefa39efp-12, t[u]);  // r
    }
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(t[u], 0.5, 1.0);
#pragma unroll
    for (int u = 0; u < N; ++u) p[u] = fma(p[u], t[u], 1.0);
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int m = __double2loint(sft[u]);
        const double v = tab[m & (kExpTab - 1)] * p[u];
        t[u] = __hiloint2double(__double2hiint(v) + ((m >> 11) << 20), __double2loint(v));
    }
}

// Running product of positive doubles as (mantissa in [1,2), exponent sum): sum of logs for one
// DMUL per term instead of a log() (about 40 FP64 instructions) per node.
struct LogProduct {
    double m = 1.0;
    long long e = 0;
    // v > 0; anything that is not a positive normal number (the caller flags those tiles for the exact
    // path) or ok == false counts as 1
    __device__ __forceinline__ void mul(double v, bool ok) {
        int hi = __double2hiint(v);
        int lo = __double2loint(v);
        const bool use = ok && (unsigned)((hi >> 20) - 1) < 2046u;
        hi = use ? hi : 0x3ff00000;
        lo = use ? lo : 0;
        e += (hi >> 20) - 1023;
        m *= __hiloint2double((hi & 0x000fffff) | 0x3ff00000, lo);
        const int mh = __double2hiint(m);  // m in [1,4): fold its exponent back
        e += (mh >> 20) - 1023;
        m = __hiloint2double((mh & 0x000fffff) | 0x3ff00000, __double2loint(m));
    }
    __device__ __forceinline__ double log_value() const { return log(m) + (double)e * 0.693147180559945309417; }
};

// feature f of the node's row: 1/sum, x_j/sum, x_a*x_b/sum (packed upper triangle), 0 on padding
template <int D, int POS>
__device__ __forceinline__ double y_feature(const double (&x)[D], const double (&xs)[D], double inv) {
    constexpr int F = n_stat_features(D);
    if constexpr (POS >= F) {
        return 0.0;
    } else if constexpr (POS == 0) {
        return inv;
    } else if constexpr (POS <= D) {
        return xs[POS - 1];
    } else {
        constexpr int r = POS - 1 - D;
        return xs[tri_row_of(r, D)] * x[tri_col_of(r, D)];
    }
}
template <int D, int... Fs>
__device__ __forceinline__ void write_y_rows(unsigned char *yb, const uint32_t (&colo)[8], const double (&x)[D],
                                             const double (&xs)[D], double inv, std::integer_sequence<int, Fs...>) {
    ((*reinterpret_cast<double *>(yb + colo[Fs & 7] + Fs * 256) = y_feature<D, Fs>(x, xs, inv)), ...);
}

// Shape of the kernel for D features and NK8 8-state tiles.  These functions are also what
// estep_bulk_supported (kernels_b3.cu) evaluates at run time, so the launch chain and the host's choice of
// kernel agree by construction.
constexpr int kYSlots = 2;  // feature-row slots per consumer
constexpr size_t kSmemMax = 227 * 1024;
constexpr int bulk_nt(int D) { return (n_stat_features(D) + 7) / 8; }  // 8-feature tiles
constexpr size_t bulk_smem_bytes(int D, int NK8, int P) {
    return (size_t)P * (8 * NK8 * 256) + (size_t)kCons * kYSlots * (8 * bulk_nt(D) * 256) + kExpTab * 8 +
           (3 * (size_t)P + kCons * kYSlots) * 8 + (size_t)P * 3 * 8 + 256;
}
// as many producer warps as shared memory and registers allow: the per-node work is latency bound
constexpr int bulk_producers(int D, int NK8) {
    return bulk_smem_bytes(D, NK8, 12) <= kSmemMax ? 12 : (bulk_smem_bytes(D, NK8, 8) <= kSmemMax ? 8 : 4);
}
// the consumer's NK8 x NT accumulator tiles (two doubles per lane each) fit its registers
constexpr bool bulk_acc_fits(int D, int NK8) { return NK8 * bulk_nt(D) * 2 <= 64; }
constexpr bool bulk_smem_fits(int D, int NK8) { return bulk_smem_bytes(D, NK8, bulk_producers(D, NK8)) <= kSmemMax; }

template <int D, int NK8>
struct BulkCfg {
    static constexpr int F = n_stat_features(D);
    static constexpr int NT = bulk_nt(D);
    static constexpr int KP = 8 * NK8, FP = 8 * NT;
    static constexpr int YS = kYSlots;
    static constexpr int E_BYTES = KP * 256, Y_BYTES = FP * 256;
    static constexpr int P = bulk_producers(D, NK8);
};
// register budgets after setmaxnreg (4 consumers + P producers share 2048 per lane column)
template <int P, bool SMALL>
struct RegBudget {
    // P = 12: 112 / 168 for a large accumulator tile, 120 / 152 for a small one (NK8*NT <= 12)
    static constexpr int prod = P == 12 ? (SMALL ? 120 : 112) : (P == 8 ? 160 : 168);
    static constexpr int cons = P == 12 ? (SMALL ? 152 : 168) : (P == 8 ? 184 : 168);
    static constexpr bool adjust = P == 12 || P == 8;  // P = 4: every warp keeps the launch allocation
};

// Row geometry of a dense region in the reference's node order (utility.py:2310-2317): node id -> (row x,
// offset c within the row, row length L).  kind 1: upper triangle of a B-bin window, row x holds the
// columns x..B-1 (L = B - x); kind 0: n1 x n2 rectangle (L = n2).
__device__ __forceinline__ void grid_locate(int kind, long long n2, long long gid, int &x, int &c, int &L) {
    if (kind == 0) {
        const long long xx = gid / n2;
        x = (int)xx;
        c = (int)(gid - xx * n2);
        L = (int)n2;
    } else {
        const double bf = (double)n2 + 0.5;
        long long xx = (long long)(bf - sqrt(bf * bf - 2.0 * (double)gid));
        if (xx < 0) xx = 0;
        if (xx > n2 - 1) xx = n2 - 1;
        auto start = [&](long long r) { return r * n2 - (r * (r - 1)) / 2; };
        while (xx > 0 && start(xx) > gid) --xx;
        while (xx < n2 - 1 && start(xx + 1) <= gid) ++xx;
        x = (int)xx;
        c = (int)(gid - start(xx));
        L = (int)(n2 - xx);
    }
}

template <int D, int NK8, int P, bool GRID, int KR>
__global__ void __launch_bounds__(32 * (kCons + P), 1) estep_bulk_kernel(EstepArgs a) {
    using C = BulkCfg<D, NK8>;
    constexpr int F = C::F, NT = C::NT, KP = C::KP, FP = C::FP, YS = C::YS;
    constexpr int E_BYTES = C::E_BYTES, Y_BYTES = C::Y_BYTES;
    constexpr int PPC = P / kCons;  // producers per consumer
    using RB = RegBudget<P, (NK8 * NT <= 12)>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // rows must start on 256-byte boundaries (the swizzle is an XOR on address bits 5-7)
    unsigned char *sbase = smem_raw + ((256u - (smem_u32(smem_raw) & 255u)) & 255u);
    unsigned char *ybase = sbase + (size_t)P * E_BYTES;
    double *tab = reinterpret_cast<double *>(ybase + (size_t)kCons * YS * Y_BYTES);
    uint64_t *bars = reinterpret_cast<uint64_t *>(tab + kExpTab);
    uint64_t *full = bars, *efree = bars + P, *landed = bars + 2 * P, *yfree = bars + 3 * P;
    double *cost_slots = reinterpret_cast<double *>(bars + 3 * P + kCons * YS);  // [P][3] per-producer cost sums
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int p = 0; p < 3 * P + kCons * YS; ++p) mbar_init(bars + p, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int j = threadIdx.x; j < kExpTab; j += blockDim.x) tab[j] = exp((double)j * (0.693147180559945309417 / kExpTab));
    __syncthreads();

    const int K = a.K, W = a.W;
    const int64_t n = a.n, ld = a.ld;
    const int64_t n_tiles = (n + kTile - 1) / kTile;
    const int64_t tile_stride_g = (int64_t)gridDim.x * P;
    const int KF = K * F;

    if (warp >= kCons) {
        // =============================== PRODUCER ===============================
        if constexpr (RB::adjust) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(RB::prod));
        const int p = warp - kCons;
        const int c = p % kCons;
        unsigned char *eb = sbase + (size_t)p * E_BYTES;
        // column of this lane in a row r: lane ^ ((r % 8) * 4); one byte offset per r % 8
        uint32_t colo[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) colo[q] = (uint32_t)((lane ^ (q << 2)) << 3);
        auto erow = [&](int r) -> double * {  // compile-time row of the E buffer
            return reinterpret_cast<double *>(eb + colo[r & 7] + r * 256);
        };
        auto dyn_off = [&](int r) -> uint32_t { return (uint32_t)((r << 8) + ((lane ^ ((r & 7) << 2)) << 3)); };
        const bool weighted = a.estimate_type == 3;
        const double beta = a.beta;
        double c_pair = 0.0, c_un = 0.0;
        LogProduct pwn_prod;  // product over this lane's nodes of the soft-max of -pp at the node's label
        int bad_any = 0;
        int j = 0;
        // implicit grid: row / offset / row length of the first node of this producer's current tile
        int gx = 0, gc = 0, gL = 1;
        const bool tri = a.grid_kind != 0;
        if (GRID) {
            const int64_t T0 = (int64_t)blockIdx.x * P + p;
            if (T0 < n_tiles) grid_locate(a.grid_kind, a.grid_n2, a.own_start_gid + T0 * kTile, gx, gc, gL);
        }
        // ---- neighbour data of tile T, loaded at the top of tile T
        int li = 0;
        int lab[kFastSlots];
        double gw[kFastSlots];   // g_s = exp(beta*w_s) (precomputed, 1 if the slot is empty)
        double ws[kFastSlots];   // edge weight as the pairwise cost counts it (0 if the slot is empty)
        int jid[GRID ? 1 : kFastSlots];  // explicit slots: neighbour ids (labels gathered at the top of the tile)
        double rmax = 0.0;
        auto load_neighbours = [&](int64_t T) {
            const int64_t i_raw = T * kTile + lane;
            const bool valid = i_raw < n;
            const int64_t i = valid ? i_raw : n - 1;
            if constexpr (GRID) {
                // this lane's node: walk from the tile's first node to its row
                int xl = gx, cl = gc + lane, Ll = gL;
                while (cl >= Ll && Ll > 0) {
                    cl -= Ll;
                    ++xl;
                    Ll = tri ? Ll - 1 : Ll;
                }
                const int rows = (int)a.grid_rows;
                const bool nn8 = a.grid_nn == 8;
                const bool up = valid && xl > 0, down = valid && xl < rows - 1;
                const bool left = valid && cl > 0, right = valid && cl < Ll - 1;
                const int dN = tri ? -Ll : -(int)a.grid_n2;      // (x-1, y)
                const int dS = tri ? Ll - 1 : (int)a.grid_n2;    // (x+1, y)
                // neighbours in ascending id: NW, N, NE, W, E, SW, S, SE; the edge weight lives with the
                // edge's forward end (slot 0 right, 1 lower left, 2 lower, 3 lower right)
                const bool v[kFastSlots] = {nn8 && up && (tri || left), up, nn8 && up && right, left, right,
                                            nn8 && down && (tri ? cl >= 2 : left), down && (tri ? cl >= 1 : true),
                                            nn8 && (tri ? right : (down && right))};
                const int dl[kFastSlots] = {dN - 1, dN, dN + 1, -1, 1, dS - 1, dS, dS + 1};
                const int fs[kFastSlots] = {3, 2, 1, 0, 0, 1, 2, 3};
                const int64_t iw = a.own_offset + i;
                li = a.labels[iw];
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) {
                    const int64_t at = iw + (s < 4 ? dl[s] : 0);  // backward edges: the neighbour holds the weight
                    const double2 wg = v[s] ? a.fwd_wg[fs[s] * a.ldw + at] : make_double2(0.0, 1.0);
                    ws[s] = weighted ? wg.x : (v[s] ? 1.0 : 0.0);
                    gw[s] = wg.y;
                }
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) lab[s] = v[s] ? a.labels[iw + dl[s]] : -1;
                // advance the tile origin to this producer's next tile
                const int64_t step = tile_stride_g * kTile;
                if (tri) {
                    int64_t cc = (int64_t)gc + step;
                    int guard = 0;
                    while (cc >= gL && gL > 0 && guard < 48) {
                        cc -= gL;
                        ++gx;
                        --gL;
                        ++guard;
                    }
                    gc = (int)cc;
                    if (cc >= gL && T + tile_stride_g < n_tiles)  // short rows near the tip: closed form
                        grid_locate(a.grid_kind, a.grid_n2, a.own_start_gid + (T + tile_stride_g) * kTile, gx, gc, gL);
                } else {
                    const int64_t cc = (int64_t)gc + step;
                    gx += (int)(cc / gL);
                    gc = (int)(cc % gL);
                }
            } else {
                const int32_t *pid = a.nbr_id + i;
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) {
                    jid[s] = s < W ? *pid : -1;
                    pid += ld;
                }
                li = a.labels[a.own_offset + i];
                const double *pw = a.nbr_w + i;
                const double *pg = a.nbr_g + i;
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) {
                    // an empty slot stores weight 0; unweighted estimates count 1 per edge
                    ws[s] = s < W ? (weighted ? *pw : (jid[s] >= 0 ? 1.0 : 0.0)) : 0.0;
                    gw[s] = s < W ? *pg : 1.0;
                    pw += ld;
                    pg += ld;
                }
            }
            rmax = a.rowmax[i];
        };
        for (int64_t T = (int64_t)blockIdx.x * P + p; T < n_tiles; T += tile_stride_g, ++j) {
            const int64_t i_raw = T * kTile + lane;
            const bool valid = i_raw < n;
            const int64_t i = valid ? i_raw : n - 1;
            {   // pull towards L2: this producer's next tile (log-likelihood, features) and the
                // neighbour data of the tile after that
                const int64_t T2 = T + tile_stride_g;
                if (T2 < n_tiles) {
                    const int64_t i2 = T2 * kTile;
                    if (lane == 0) bulk_prefetch_l2(a.logp + T2 * (KP * 32), KP * 256);
                    if (lane < 2 * D) prefetch_l2(a.X_soa + (lane >> 1) * ld + i2 + (lane & 1) * 16);
                }
                const int64_t T3 = T2 + tile_stride_g;
                if (T3 < n_tiles) {
                    const int64_t i3 = T3 * kTile;
                    if (GRID) {  // 4 forward slots x 32 nodes x 16 bytes = 4 lines per slot
                        if (lane >= 16) prefetch_l2(a.fwd_wg + ((lane - 16) >> 2) * a.ldw + a.own_offset + i3 + ((lane - 16) & 3) * 8);
                    } else {
                        if (lane < 2 * W) prefetch_l2(a.nbr_w + (lane >> 1) * ld + i3 + (lane & 1) * 16);
                        if (lane >= 16 && lane - 16 < 2 * W)
                            prefetch_l2(a.nbr_g + ((lane - 16) >> 1) * ld + i3 + (lane & 1) * 16);
                        if (lane < W) prefetch_l2(a.nbr_id + lane * ld + i3);
                    }
                    if (lane == 15) prefetch_l2(a.rowmax + i3);
                }
            }
            load_neighbours(T);
            if constexpr (!GRID) {
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) lab[s] = jid[s] >= 0 ? a.labels[jid[s]] : -1;
            }
            double pc = 0.0;   // sum over the incident edges of V[l_nbr, l_i] * w
            int all_neg = -1;  // sign bit stays set while no slot holds a neighbour
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                all_neg &= lab[s];
                pc += lab[s] != li ? ws[s] : 0.0;
            }
            pc *= beta;
            if (all_neg < 0) {  // isolated node: pp = V[label] unweighted (phylo_hmrf.py:421-423)
                lab[0] = li;
                gw[0] = a.exp_beta;
            }
            // byte offsets of row label_s in this lane's UNswizzled column (0xffff: empty slot), two per
            // register.  A lane keeps to its own bank pair whatever the row, so the label-indexed scratch
            // accesses below are conflict free; the swizzled offset the consumer's layout needs is
            // raw ^ ((raw >> 3) & 0xe0).
            uint32_t offp[kFastSlots / 2];
#pragma unroll
            for (int s = 0; s < kFastSlots; s += 2) {
                const uint32_t o0 = lab[s] >= 0 ? (uint32_t)((lab[s] << 8) + (lane << 3)) : 0xffffu;
                const uint32_t o1 = lab[s + 1] >= 0 ? (uint32_t)((lab[s + 1] << 8) + (lane << 3)) : 0xffffu;
                offp[s / 2] = o0 | (o1 << 16);
            }
            const uint32_t off_li = dyn_off(li);
            const uint32_t raw_li = (uint32_t)((li << 8) + (lane << 3));
            const double rmax_t = rmax;
            // ---- the E buffer is free once the consumer has released the previous tile.  First use:
            // scratch for G_k -- ones, then g_s multiplied into G[label_s] slot by slot
            // (exp(a)exp(b) = exp(a+b): no duplicate-label bookkeeping).  The host only selects this
            // kernel when |beta| * W * max|w| < 100, so the products stay finite.
            if (j > 0) mbar_wait(efree + p, (uint32_t)((j - 1) & 1));
            // (only the rows the neighbours' labels and the node's own label select are ever read)
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                const uint32_t o = (offp[s / 2] >> (16 * (s & 1))) & 0xffffu;
                if (o != 0xffffu) *reinterpret_cast<double *>(eb + o) = 1.0;
            }
            *reinterpret_cast<double *>(eb + raw_li) = 1.0;
            double qs = 0.0;  // sum_k G_k - K
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                const uint32_t o = (offp[s / 2] >> (16 * (s & 1))) & 0xffffu;
                if (o != 0xffffu) {
                    double *gp = reinterpret_cast<double *>(eb + o);
                    const double g_old = *gp;
                    const double g_new = g_old * gw[s];
                    *gp = g_new;
                    qs += g_new - g_old;
                }
            }
            const double g_li = *reinterpret_cast<double *>(eb + raw_li);
            // ---- second use: the log-likelihood tile, one bulk copy
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                mbar_expect_tx(landed + p, KP * 256);
                bulk_g2s(eb, a.logp + T * (KP * 32), KP * 256, landed + p);
            }
            const double qsum = (double)K + qs;
            // soft-max of -pp at the node's own label: exp(S_li) / sum_k exp(S_k)
            const double pwn = fma(g_li, fast_rcp(qsum), 1e-16);
            mbar_wait(landed + p, (uint32_t)(j & 1));
            const double lp_li = *reinterpret_cast<double *>(eb + off_li);
            // soft-max shift = max(logp_li, max_k logp_k - 598): overflow-free for any labels
            const double shift = valid ? fmax(lp_li, rmax_t - 598.0) : 1.0e300;
            double esum = 0.0;
#pragma unroll 1
            for (int cc = 0; cc < NK8 - 1; ++cc) {  // not unrolled: the instruction cache is shared by all warps
                double tb[8];
                unsigned char *ec = eb + cc * 2048;
#pragma unroll
                for (int u = 0; u < 8; ++u) tb[u] = *reinterpret_cast<double *>(ec + colo[u] + u * 256) - shift;
                exp_tab<8>(tb, tab);
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    esum += tb[u];
                    *reinterpret_cast<double *>(ec + colo[u] + u * 256) = tb[u];
                }
            }
            {   // last 8-state chunk: KR live rows; the rest are padding states, whose rows arrive from HBM as
                // 0.0 -- already the zero weight the statistics product needs (common.cuh logp_rows)
                double tb[KR];
                unsigned char *ec = eb + (NK8 - 1) * 2048;
#pragma unroll
                for (int u = 0; u < KR; ++u) tb[u] = *reinterpret_cast<double *>(ec + colo[u] + u * 256) - shift;
                exp_tab<KR>(tb, tab);
#pragma unroll
                for (int u = 0; u < KR; ++u) {
                    esum += tb[u];
                    *reinterpret_cast<double *>(ec + colo[u] + u * 256) = tb[u];
                }
            }
            // the node's features: in flight while the neighbour factors are applied
            double x[D];
            const double *px = a.X_soa + i;
#pragma unroll
            for (int jx = 0; jx < D; ++jx) {
                x[jx] = *px;
                px += ld;
            }
            // e_k *= g_s for every neighbour slot in turn (a label met twice is multiplied twice: the product)
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                const uint32_t o = (offp[s / 2] >> (16 * (s & 1))) & 0xffffu;
                if (o != 0xffffu) {
                    double *ep = reinterpret_cast<double *>(eb + (o ^ ((o >> 3) & 0xe0u)));
                    const double e_old = *ep;
                    const double e_new = e_old * gw[s];
                    *ep = e_new;
                    esum += e_new - e_old;
                }
            }
            const bool bad = !(esum <= DBL_MAX) || !(qsum <= DBL_MAX) || !(esum > 0.0);
            bad_any |= (bad && valid) ? 1 : 0;
            const double inv = valid ? fast_rcp(esum) : 0.0;
            if (valid) {
                c_pair += all_neg < 0 ? 0.0 : pc;
                c_un += lp_li;
            }
            pwn_prod.mul(pwn, valid);
            if (a.post_soa != nullptr) {
                if (valid) {
#pragma unroll 1
                    for (int q = 0; q < K; ++q)
                        a.post_soa[q * ld + i] = *reinterpret_cast<double *>(eb + dyn_off(q)) * inv;
                }
            }
            // ---- feature rows into the next Y slot of this producer's consumer (tile order)
            const int m = p / kCons + PPC * j;  // index among the consumer's tiles
            const int ys = m % YS;
            unsigned char *yb = ybase + (size_t)(c * YS + ys) * Y_BYTES;
            if (m >= YS) mbar_wait(yfree + c * YS + ys, (uint32_t)((m / YS - 1) & 1));
            {   // row 0: 1/sum; rows 1..D: x_a/sum; then the packed products, one scaled feature live at a time
                auto yrow = [&](int f) -> double * { return reinterpret_cast<double *>(yb + colo[f & 7] + f * 256); };
                *yrow(0) = inv;
                int f2 = 1 + D;
#pragma unroll
                for (int ja = 0; ja < D; ++ja) {
                    const double xa = x[ja] * inv;
                    *yrow(1 + ja) = xa;
#pragma unroll
                    for (int jb = ja; jb < D; ++jb) *yrow(f2++) = xa * x[jb];
                }
#pragma unroll
                for (int f = F; f < FP; ++f) *yrow(f) = 0.0;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(full + p);
        }
        if (bad_any) atomicOr(a.flags, 1);
        double c_pwn = pwn_prod.log_value();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c_pair += __shfl_xor_sync(0xffffffffu, c_pair, o);
            c_pwn += __shfl_xor_sync(0xffffffffu, c_pwn, o);
            c_un += __shfl_xor_sync(0xffffffffu, c_un, o);
        }
        if (lane == 0) {   // this producer's cost sums; added up in producer order after the block barrier
            cost_slots[3 * p + 0] = c_pair;
            cost_slots[3 * p + 1] = c_pwn;
            cost_slots[3 * p + 2] = c_un;
        }
    } else {
        // =============================== CONSUMER ===============================
        if constexpr (RB::adjust) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(RB::cons));
        const int c = warp;
        const int g = lane >> 2, t = lane & 3;
        double acc[NK8][NT][2];
#pragma unroll
        for (int kt = 0; kt < NK8; ++kt)
#pragma unroll
            for (int ft = 0; ft < NT; ++ft) acc[kt][ft][0] = acc[kt][ft][1] = 0.0;
        // byte offset of (row 8*tile + g, node 4*ns + t) in a buffer:
        //   ((g*256 + t*8) ^ (g << 5)) ^ (ns << 5)  +  tile * 2048
        const uint32_t pk = (uint32_t)((g << 8) + (t << 3)) ^ (uint32_t)(g << 5);
        int cnt[PPC];
#pragma unroll
        for (int q = 0; q < PPC; ++q) {
            const int64_t gidx = (int64_t)blockIdx.x * P + (c + q * kCons);
            cnt[q] = n_tiles > gidx ? (int)((n_tiles - gidx - 1) / tile_stride_g + 1) : 0;
        }
        int m = 0;  // tiles consumed so far: the Y slots are claimed in this order
        for (int j = 0; j < cnt[0]; ++j) {  // cnt[0] >= cnt[q] for every q
#pragma unroll 1
            for (int q = 0; q < PPC; ++q) {
                if (j < cnt[q]) {
                    const int p = c + q * kCons;
                    const int ys = m % YS;
                    const unsigned char *eb = sbase + (size_t)p * E_BYTES;
                    const unsigned char *yb = ybase + (size_t)(c * YS + ys) * Y_BYTES;
                    mbar_wait(full + p, (uint32_t)(j & 1));
#pragma unroll 2
                    for (int ns = 0; ns < kTile / 4; ++ns) {
                        double av[NK8], bv[NT];
                        const uint32_t o = pk ^ (uint32_t)(ns << 5);
#pragma unroll
                        for (int kt = 0; kt < NK8; ++kt) av[kt] = *reinterpret_cast<const double *>(eb + o + kt * 2048);
#pragma unroll
                        for (int ft = 0; ft < NT; ++ft) bv[ft] = *reinterpret_cast<const double *>(yb + o + ft * 2048);
#pragma unroll
                        for (int kt = 0; kt < NK8; ++kt)
#pragma unroll
                            for (int ft = 0; ft < NT; ++ft) dmma_8x8x4(acc[kt][ft][0], acc[kt][ft][1], av[kt], bv[ft]);
                    }
                    __syncwarp();
                    if (lane == 0) {
                        mbar_arrive(efree + p);
                        mbar_arrive(yfree + c * YS + ys);
                    }
                    ++m;
                }
            }
        }
        // every tile of this consumer is consumed, so its two Y slots are free: the K x F partial sums go there
        // (2 * Y_BYTES = NT * 4096 bytes >= K * F * 8 for NK8 <= 8), dense [K][F]
        double *part = reinterpret_cast<double *>(ybase + (size_t)(c * YS) * Y_BYTES);
#pragma unroll
        for (int kt = 0; kt < NK8; ++kt) {
            const int k = 8 * kt + g;
#pragma unroll
            for (int ft = 0; ft < NT; ++ft)
#pragma unroll
                for (int jj = 0; jj < 2; ++jj) {
                    const int f = 8 * ft + 2 * t + jj;
                    if (k < K && f < F) part[k * F + f] = acc[kt][ft][jj];
                }
        }
    }
    // One block-wide barrier at a single call site (both roles fall through to it), then the consumers'
    // partial sums are added in consumer order and the producers' cost sums in producer order: the result does not
    // depend on timing (bit-reproducible), and the per-CTA partials go out for estep_finalize_kernel.
    static_assert((size_t)YS * Y_BYTES >= (size_t)KP * FP * 8, "partial sums must fit the consumer's Y slots");
    __syncthreads();
    double *out = a.partials + (size_t)blockIdx.x * (KF + 3);
    for (int e0 = threadIdx.x; e0 < KF; e0 += blockDim.x) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < kCons; ++w) v += reinterpret_cast<const double *>(ybase + (size_t)(w * YS) * Y_BYTES)[e0];
        out[e0] = v;
    }
    if (threadIdx.x < 3) {
        double v = 0.0;
        for (int w = 0; w < P; ++w) v += cost_slots[3 * w + threadIdx.x];
        out[KF + threadIdx.x] = v;
    }
}

// a shape that estep_bulk_supported rejects reached the launcher: the caller's error, never a fall-back
int bulk_unsupported(const EstepArgs &a) {
    set_error("estep_bulk_kernel: no instantiation for n_features=" + std::to_string(a.D) +
              ", n_states=" + std::to_string(a.K));
    return PHMRF_E_UNSUPPORTED;
}

template <int D, int NK8, int P, int KR>
int launch_bulk_pk(const EstepArgs &a, int sm_count, cudaStream_t s) {
    const size_t smem = bulk_smem_bytes(D, NK8, P);
    const int64_t n_tiles = (a.n + kTile - 1) / kTile;
    int64_t want = (n_tiles + P - 1) / P;
    const int grid = (int)(want < sm_count ? (want < 1 ? 1 : want) : sm_count);
    auto kern = a.fwd_wg != nullptr ? estep_bulk_kernel<D, NK8, P, true, KR> : estep_bulk_kernel<D, NK8, P, false, KR>;
    PHMRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 32 * (kCons + P), smem, s>>>(a);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    return launch_estep_finalize(a.partials, grid, a.K, D, a.stats_out, s);
}

// KR: states of the last 8-state chunk that are evaluated (K's remainder rounded up to even); the
// other rows of that chunk are padding and get zero weight without an exp()
template <int D, int NK8, int P>
int launch_bulk_p(const EstepArgs &a, int sm_count, cudaStream_t s) {
    switch ((a.K - 8 * (NK8 - 1) + 1) & ~1) {
        case 2: return launch_bulk_pk<D, NK8, P, 2>(a, sm_count, s);
        case 4: return launch_bulk_pk<D, NK8, P, 4>(a, sm_count, s);
        case 6: return launch_bulk_pk<D, NK8, P, 6>(a, sm_count, s);
        default: return launch_bulk_pk<D, NK8, P, 8>(a, sm_count, s);
    }
}

template <int D, int NK8>
int launch_bulk(const EstepArgs &a, int sm_count, cudaStream_t s) {
    if constexpr (!bulk_acc_fits(D, NK8) || !bulk_smem_fits(D, NK8)) {
        return bulk_unsupported(a);
    } else {
        return launch_bulk_p<D, NK8, BulkCfg<D, NK8>::P>(a, sm_count, s);
    }
}

template <int D>
int launch_bulk_d(const EstepArgs &a, int sm_count, cudaStream_t s) {
    switch ((a.K + 7) / 8) {
        case 1: return launch_bulk<D, 1>(a, sm_count, s);
        case 2: return launch_bulk<D, 2>(a, sm_count, s);
        case 3: return launch_bulk<D, 3>(a, sm_count, s);
        case 4: return launch_bulk<D, 4>(a, sm_count, s);
        case 5: return launch_bulk<D, 5>(a, sm_count, s);
        default: return bulk_unsupported(a);
    }
}

}  // namespace

// one translation unit per range of feature counts (kernels_b3.cu, kernels_b3_d58.cu, kernels_b3_d9c.cu):
// the instantiations compile in parallel
int PHMRF_B3_ENTRY(const EstepArgs &a, int sm_count, cudaStream_t s) {
    switch (a.D) {
#define PHMRF_CASE(DD) \
    case DD:           \
        return launch_bulk_d<DD>(a, sm_count, s);
        PHMRF_CASE(PHMRF_B3_D0) PHMRF_CASE(PHMRF_B3_D0 + 1) PHMRF_CASE(PHMRF_B3_D0 + 2) PHMRF_CASE(PHMRF_B3_D0 + 3)
#undef PHMRF_CASE
    }
    return bulk_unsupported(a);
}

}  // namespace phmrf
