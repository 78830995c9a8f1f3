// Phase B of the Phylo-HMRF E-step on sm_100a: neighbour-weighted pairwise potential,
// posteriors, the cost scalars and the M-step sufficient statistics in ONE pass over the
// nodes (pp, the posteriors and the per-node features are never materialised in HBM).
//
// Reference arithmetic: _pairwise_compare/_pairwise_compareLocal (phylo_hmrf.py:398-436),
// _compute_posteriors_graph (:334-355), _compute_cost_v1 (:374-396),
// _pairwise_compare_ensemble/_single (:438-468), statistics triple (:311-314).
//
// Structure.  A warp owns 32 consecutive nodes per step (lane = node) and runs two phases:
//   node phase  lane-private: gather neighbour labels, scatter beta*w into a shared-memory
//               row (one row per node), soft-max over the K states, cost terms, and the
//               per-node feature row y = (1, x, x (x) x packed) / normaliser.
//   stat phase  S[k][f] += sum_n e[n][k] * y[n][f] is a (K x 32) x (32 x F) product whose
//               K*F accumulators are spread over the lanes of the warp as TK x TF register
//               tiles; rows are read back from shared memory as broadcast LDS.128.
// Accumulators live in registers for the whole kernel; block partials are reduced in a
// fixed order (deterministic) and a final kernel folds them and unpacks the symmetric
// scatter into the reference's [K], [K,d], [K,d,d] layout.
#include <cstdlib>

#include "estep_common.cuh"

namespace phmrf {

using namespace estep;

namespace {

template <int D, int TK, int TF>
__global__ void __launch_bounds__(kThreads, 1) estep_kernel(EstepArgs a, int nkt_total, int kt_begin, int nkt_pass,
                                                             int rsp, int first_pass) {
    using C = Cfg<D, TK, TF>;
    constexpr int F = C::F, TKs = C::TKs, TFs = C::TFs, NFT = C::NFT, RSY = C::RSY;
    extern __shared__ __align__(16) double smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    double *Ps = smem + (size_t)warp * 32 * (rsp + RSY);
    double *Ys = Ps + 32 * rsp;
    double *Prow = Ps + lane * rsp;
    double *Yrow = Ys + lane * RSY;

    // lane -> (node subset, k tile, f tile) for the stat phase
    const int tiles = nkt_pass * NFT;
    const int NS = 32 / tiles;
    const int sub = lane / tiles;
    const int tl = lane - sub * tiles;
    const int ktl = tl / NFT, ft = tl - ktl * NFT;
    const bool lane_active = sub < NS && (kt_begin + ktl) < nkt_total;
    const int kt = lane_active ? kt_begin + ktl : kt_begin;

    double acc[TK][TF];
#pragma unroll
    for (int i = 0; i < TK; ++i)
#pragma unroll
        for (int j = 0; j < TF; ++j) acc[i][j] = 0.0;
    double c_pair = 0.0, c_pwn = 0.0, c_un = 0.0;

    const int K = a.K, W = a.W;
    const int KP = logp_rows(K);
    const int64_t n = a.n, ld = a.ld;
    const int64_t n_tiles = (n + 31) >> 5;
    const int64_t warp_global = (int64_t)blockIdx.x * wpb + warp;
    const int64_t warp_stride = (int64_t)gridDim.x * wpb;
    const bool weighted = a.estimate_type == 3;
    const double beta = a.beta;
    const bool fast_ok = a.potts && W <= kFastSlots && a.pp_soa == nullptr;

    for (int64_t t = warp_global; t < n_tiles; t += warp_stride) {
        const int64_t i_raw = (t << 5) + lane;
        const bool valid = i_raw < n;
        const int64_t i = valid ? i_raw : n - 1;

        // pull the next tile of this warp towards L2 while this one is processed
        {
            const int64_t t2 = t + warp_stride;
            if (t2 < n_tiles) {
                const int64_t i2 = t2 << 5;
                for (int q = lane; q < 2 * K; q += 32) prefetch_l2(a.logp + (t2 * KP + (q >> 1)) * 32 + (q & 1) * 16);
                for (int q = lane; q < 2 * D; q += 32) prefetch_l2(a.X_soa + (q >> 1) * ld + i2 + (q & 1) * 16);
                for (int q = lane; q < 2 * W; q += 32) prefetch_l2(a.nbr_w + (q >> 1) * ld + i2 + (q & 1) * 16);
                for (int q = lane; q < W; q += 32) prefetch_l2(a.nbr_id + q * ld + i2);
            }
        }

        const int li = a.labels[a.own_offset + i];
        const int pos_li = (li / TK) * TKs + (li % TK);
        const double lp_li = a.logp[lp_index(li, i, KP)];

        // ---------------- node phase ----------------
        double pc = 0.0, pwn_log = 0.0, esum = 0.0;
        bool need_exact = !fast_ok;
        if (fast_ok) {
            // Potts compatibility, <= 8 neighbour slots: everything neighbour-related stays in
            // registers.  With S_c = sum of beta*w over the neighbours carrying label c,
            //   pp_k = wtot - S_k,   exp(logp_k - pp_k - shift) = exp(logp_k - c0) * exp(S_k),
            // c0 = logp_li + S_li, so the K-wide pass needs no per-state neighbour data and the
            // <= 8 distinct neighbour labels are patched afterwards with f_c = exp(S_c).
            int lab[kFastSlots];
            double sw[kFastSlots];
            bool live[kFastSlots];
            {
                int jid[kFastSlots];
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) jid[s] = s < W ? a.nbr_id[s * ld + i] : -1;
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) lab[s] = jid[s] >= 0 ? a.labels[jid[s]] : -1 - s;
#pragma unroll
                for (int s = 0; s < kFastSlots; ++s) {
                    sw[s] = 0.0;
                    if (jid[s] >= 0) sw[s] = weighted ? beta * a.nbr_w[s * ld + i] : beta;
                    live[s] = jid[s] >= 0;
                }
            }
            bool any_nbr = false;
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                any_nbr |= live[s];
                pc += (live[s] && lab[s] != li) ? sw[s] : 0.0;
            }
            if (!any_nbr) {  // isolated node: pp = V[label] unweighted (phylo_hmrf.py:421-423)
                lab[0] = li;
                sw[0] = beta;
                live[0] = true;
            }
            // fold duplicate labels into their first occurrence
#pragma unroll
            for (int s = 1; s < kFastSlots; ++s)
#pragma unroll
                for (int q = 0; q < s; ++q) {
                    const bool dup = live[s] && live[q] && lab[q] == lab[s];
                    sw[q] += dup ? sw[s] : 0.0;
                    live[s] = live[s] && !dup;
                }
            double s_li = 0.0, fsum = 0.0, f_li = 1.0;
            double f[kFastSlots];
            int m = 0;
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                f[s] = 1.0;
                if (__any_sync(0xffffffffu, live[s])) {
                    const double e = exp_sm(sw[s]);
                    if (live[s]) {
                        f[s] = e;
                        fsum += e;
                        ++m;
                        if (lab[s] == li) {
                            s_li = sw[s];
                            f_li = e;
                        }
                    }
                }
            }
            // soft-max of -pp at the node's own label: exp(S_li) / (sum_c exp(S_c) + (K - m))
            pwn_log = log(f_li / (fsum + (double)(K - m)) + 1e-16);
            const double c0 = lp_li + s_li;
#pragma unroll 2
            for (int ktile = 0; ktile < nkt_total; ++ktile) {
                double e[TKs];
#pragma unroll
                for (int ii = 0; ii < TKs; ++ii) e[ii] = 0.0;
#pragma unroll
                for (int ii = 0; ii < TK; ++ii) {
                    const int k = ktile * TK + ii;
                    if (k < K) e[ii] = a.logp[lp_index(k, i, KP)];
                }
#pragma unroll
                for (int ii = 0; ii < TK; ++ii) {
                    const int k = ktile * TK + ii;
                    e[ii] = k < K ? exp_sm(e[ii] - c0) : 0.0;
                    esum += e[ii];
                }
#pragma unroll
                for (int c = 0; c < TKs; c += 2)
                    *reinterpret_cast<double2 *>(Prow + ktile * TKs + c) = make_double2(e[c], e[c + 1]);
            }
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                if (__any_sync(0xffffffffu, live[s])) {
                    if (live[s]) {
                        const int pos = (lab[s] / TK) * TKs + (lab[s] % TK);
                        const double e_old = Prow[pos];
                        const double e_new = e_old * f[s];
                        Prow[pos] = e_new;
                        esum += e_new - e_old;
                    }
                }
            }
            const bool bad = !(esum <= DBL_MAX) || !(fsum <= DBL_MAX);
            need_exact = __any_sync(0xffffffffu, bad);
        }
        if (need_exact) {
            // General path: any compatibility matrix, any degree, exact soft-max maximum.
            double wtot = 0.0, pmin = 0.0, qsum = 1.0, pp_li;
            pc = 0.0;
            if (a.potts) {
                for (int c = 0; c < rsp; c += 2) *reinterpret_cast<double2 *>(Prow + c) = make_double2(0.0, 0.0);
                double smax = 0.0;
                int deg = 0;
                for (int s = 0; s < W; ++s) {
                    const int j = a.nbr_id[s * ld + i];
                    if (j >= 0) {
                        const int lj = a.labels[j];
                        const double bw = weighted ? beta * a.nbr_w[s * ld + i] : beta;
                        const int pos = (lj / TK) * TKs + (lj % TK);
                        const double v = Prow[pos] + bw;
                        Prow[pos] = v;
                        smax = fmax(smax, v);
                        wtot += bw;
                        pc += (lj != li) ? bw : 0.0;
                        ++deg;
                    }
                }
                if (deg == 0) {
                    wtot = beta;
                    Prow[pos_li] = beta;
                    smax = beta;
                }
                const double s_li = Prow[pos_li];
                pp_li = wtot - s_li;
                pmin = wtot - smax;
                if (first_pass) {
                    // K - m states carry pp = wtot, the m labels seen among the neighbours carry
                    // wtot - S; a counted S is flagged by flipping its sign.
                    double qs = 0.0;
                    int m = 0;
                    for (int s = 0; s < W; ++s) {
                        const int j = a.nbr_id[s * ld + i];
                        const int lj = j >= 0 ? a.labels[j] : li;
                        const int pos = (lj / TK) * TKs + (lj % TK);
                        const double v = Prow[pos];
                        if (j >= 0 && v > 0.0) {
                            qs += exp(v - smax);
                            ++m;
                            Prow[pos] = -v;
                        }
                    }
                    if (deg == 0) {
                        qs = 1.0;
                        m = 1;
                    }
                    qsum = qs + (double)(K - m) * exp(-smax);
                    pwn_log = log(exp(s_li - smax) / qsum + 1e-16);
                }
            } else {
                int deg = 0;
                for (int s = 0; s < W; ++s) deg += a.nbr_id[s * ld + i] >= 0;
                pmin = INFINITY;
                pp_li = 0.0;
                for (int k = 0; k < K; ++k) {
                    double pp = 0.0;
                    if (deg == 0) {
                        pp = a.V[li * K + k];
                    } else {
                        for (int s = 0; s < W; ++s) {
                            const int j = a.nbr_id[s * ld + i];
                            if (j >= 0) pp += a.V[a.labels[j] * K + k] * (weighted ? a.nbr_w[s * ld + i] : 1.0);
                        }
                    }
                    Prow[(k / TK) * TKs + (k % TK)] = pp;
                    pmin = fmin(pmin, pp);
                    if (k == li) pp_li = pp;
                }
                for (int s = 0; s < W; ++s) {
                    const int j = a.nbr_id[s * ld + i];
                    if (j >= 0) pc += a.V[a.labels[j] * K + li] * (weighted ? a.nbr_w[s * ld + i] : 1.0);
                }
                if (first_pass) {
                    qsum = 0.0;
                    for (int k = 0; k < K; ++k) qsum += exp(pmin - Prow[(k / TK) * TKs + (k % TK)]);
                    pwn_log = log(exp(pmin - pp_li) / qsum + 1e-16);
                }
            }
            double amax = -INFINITY;
            for (int ktile = 0; ktile < nkt_total; ++ktile) {
#pragma unroll
                for (int ii = 0; ii < TK; ++ii) {
                    const int k = ktile * TK + ii;
                    if (k < K) {
                        const double sv = Prow[ktile * TKs + ii];
                        const double pp = a.potts ? wtot - fabs(sv) : sv;
                        amax = fmax(amax, a.logp[lp_index(k, i, KP)] - pp);
                    }
                }
            }
            esum = 0.0;
            for (int ktile = 0; ktile < nkt_total; ++ktile) {
#pragma unroll
                for (int ii = 0; ii < TKs; ++ii) {
                    const int k = ktile * TK + ii;
                    double e = 0.0;
                    if (ii < TK && k < K) {
                        const double sv = Prow[ktile * TKs + ii];
                        const double pp = a.potts ? wtot - fabs(sv) : sv;
                        e = exp((a.logp[lp_index(k, i, KP)] - pp) - amax);
                        if (a.pp_soa != nullptr && first_pass && valid) a.pp_soa[k * ld + i] = pp;
                    }
                    esum += e;
                    Prow[ktile * TKs + ii] = e;
                }
            }
        }

        const double inv = valid ? 1.0 / esum : 0.0;
        if (first_pass && valid) {
            c_pair += pc;
            c_un += lp_li;
            c_pwn += pwn_log;
            if (a.post_soa != nullptr) {
                for (int ktile = 0; ktile < nkt_total; ++ktile)
#pragma unroll
                    for (int ii = 0; ii < TK; ++ii) {
                        const int k = ktile * TK + ii;
                        if (k < K) a.post_soa[k * ld + i] = Prow[ktile * TKs + ii] * inv;
                    }
            }
        }
        {
            double x[D], xs[D];
#pragma unroll
            for (int j = 0; j < D; ++j) {
                x[j] = a.X_soa[j * ld + i];
                xs[j] = x[j] * inv;
            }
            write_y_row<D, TF, TFs>(Yrow, x, xs, inv, std::make_integer_sequence<int, RSY / 2>{});
        }
        __syncwarp();

        // ---------------- stat phase ----------------
        if (lane_active) {
            const double *pb = Ps + kt * TKs;
            const double *yb = Ys + ft * TFs;
#pragma unroll 2
            for (int nn = sub; nn < 32; nn += NS) {
                double p[even_up(TK)], y[even_up(TF)];
#pragma unroll
                for (int c = 0; c < even_up(TK); c += 2) {
                    const double2 v = *reinterpret_cast<const double2 *>(pb + nn * rsp + c);
                    p[c] = v.x;
                    p[c + 1] = v.y;
                }
#pragma unroll
                for (int c = 0; c < even_up(TF); c += 2) {
                    const double2 v = *reinterpret_cast<const double2 *>(yb + nn * RSY + c);
                    y[c] = v.x;
                    y[c + 1] = v.y;
                }
#pragma unroll
                for (int ii = 0; ii < TK; ++ii)
#pragma unroll
                    for (int jj = 0; jj < TF; ++jj) acc[ii][jj] = fma(p[ii], y[jj], acc[ii][jj]);
            }
        }
        __syncwarp();
    }

    // ---------------- block reduction (fixed order => deterministic) ----------------
    __syncthreads();
    double *red = smem;  // K*F + 3 doubles
    const int KF = K * F;
    for (int e = threadIdx.x; e < KF + 3; e += blockDim.x) red[e] = 0.0;
    __syncthreads();
    for (int w = 0; w < wpb; ++w) {
        for (int s = 0; s < NS; ++s) {
            if (warp == w && sub == s && lane_active) {
#pragma unroll
                for (int ii = 0; ii < TK; ++ii) {
                    const int k = kt * TK + ii;
#pragma unroll
                    for (int jj = 0; jj < TF; ++jj) {
                        const int f = ft * TF + jj;
                        if (k < K && f < F) red[k * F + f] += acc[ii][jj];
                    }
                }
            }
            __syncthreads();
        }
    }
    // cost partial sums: warp shuffle tree, then warps in order
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        c_pair += __shfl_xor_sync(0xffffffffu, c_pair, o);
        c_pwn += __shfl_xor_sync(0xffffffffu, c_pwn, o);
        c_un += __shfl_xor_sync(0xffffffffu, c_un, o);
    }
    for (int w = 0; w < wpb; ++w) {
        if (warp == w && lane == 0) {
            red[KF + 0] += c_pair;
            red[KF + 1] += c_pwn;
            red[KF + 2] += c_un;
        }
        __syncthreads();
    }
    double *out = a.partials + (size_t)blockIdx.x * (KF + 3);
    const int k_lo = kt_begin * TK, k_hi = min(K, (kt_begin + nkt_pass) * TK);
    for (int e = threadIdx.x; e < KF + 3; e += blockDim.x) {
        if (e >= KF) {
            if (first_pass) out[e] = red[e];
        } else {
            const int k = e / F;
            if (k >= k_lo && k < k_hi) out[e] = red[e];
        }
    }
}

// Fold the per-block partials (fixed order) and unpack to post[K] | obs[K,d] | obs*obs.T[K,d,d] | 3 cost sums.
__global__ void estep_finalize_kernel(const double *__restrict__ partials, int n_blocks, int K, int D,
                                      double *__restrict__ stats_out) {
    const int F = n_stat_features(D);
    const int KF = K * F;
    const int n_out = K * (1 + D + D * D) + 3;
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += gridDim.x * blockDim.x) {
        int src;
        if (o < K) {
            src = o * F;
        } else if (o < K + K * D) {
            const int k = (o - K) / D, i = (o - K) % D;
            src = k * F + 1 + i;
        } else if (o < K + K * D + K * D * D) {
            const int r = o - K - K * D;
            const int k = r / (D * D), ij = r % (D * D);
            int i = ij / D, j = ij % D;
            if (i > j) {
                const int tmp = i;
                i = j;
                j = tmp;
            }
            src = k * F + 1 + D + (i * D - i * (i - 1) / 2 + (j - i));
        } else {
            src = KF + (o - (K + K * D + K * D * D));
        }
        double s = 0.0;
        for (int b = 0; b < n_blocks; ++b) s += partials[(size_t)b * (KF + 3) + src];
        stats_out[o] = s;
    }
}

struct Plan {
    int nkt_total, nkt_pass, n_pass, rsp, wpb, grid;
    size_t smem;
};

template <int D>
Plan make_plan(int K, int sm_count, int64_t n) {
    constexpr TileChoice tc = tile_for(D);
    using C = Cfg<D, tc.tk, tc.tf>;
    Plan p;
    p.nkt_total = (K + tc.tk - 1) / tc.tk;
    int max_kt = 32 / C::NFT;
    p.nkt_pass = p.nkt_total < max_kt ? p.nkt_total : max_kt;
    p.n_pass = (p.nkt_total + p.nkt_pass - 1) / p.nkt_pass;
    p.rsp = pad_row(p.nkt_total * C::TKs);
    size_t per_warp = (size_t)32 * (p.rsp + C::RSY) * sizeof(double);
    size_t budget = 220 * 1024;
    int wpb = (int)(budget / per_warp);
    if (wpb > 8) wpb = 8;
    p.wpb = wpb;
    size_t red_bytes = ((size_t)K * C::F + 3) * sizeof(double);
    p.smem = per_warp * (wpb > 0 ? wpb : 1);
    if (p.smem < red_bytes) p.smem = red_bytes;
    int64_t n_tiles = (n + 31) / 32;
    int64_t want = wpb > 0 ? (n_tiles + wpb - 1) / wpb : 1;
    p.grid = (int)(want < sm_count ? (want < 1 ? 1 : want) : sm_count);
    return p;
}

template <int D>
int launch_estep_d(const EstepArgs &a, int sm_count, cudaStream_t s) {
    constexpr TileChoice tc = tile_for(D);
    Plan p = make_plan<D>(a.K, sm_count, a.n);
    if (p.wpb < 1 || p.smem > 227 * 1024) {
        set_error("n_states too large for the E-step shared-memory rows");
        return PHMRF_E_UNSUPPORTED;
    }
    auto kern = estep_kernel<D, tc.tk, tc.tf>;
    PHMRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    for (int pass = 0; pass < p.n_pass; ++pass) {
        kern<<<p.grid, p.wpb * 32, p.smem, s>>>(a, p.nkt_total, pass * p.nkt_pass, p.nkt_pass, p.rsp, pass == 0);
        count_launch();
        PHMRF_CUDA(cudaGetLastError());
    }
    return launch_estep_finalize(a.partials, p.grid, a.K, D, a.stats_out, s);
}

}  // namespace

int launch_estep_finalize(const double *partials, int n_blocks, int K, int D, double *stats_out, cudaStream_t s) {
    estep_finalize_kernel<<<8, 256, 0, s>>>(partials, n_blocks, K, D, stats_out);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

// g[s][i] = exp(beta * (weighted ? w[s][i] : 1)) for occupied neighbour slots, 1 otherwise: the per-slot
// factors of the pipeline kernel for regions with an explicit graph; constant while beta and the weights are
__global__ void nbr_g_kernel(const int32_t *__restrict__ nbr_id, const double *__restrict__ nbr_w,
                             double *__restrict__ nbr_g, int64_t count, double beta, int weighted) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
        nbr_g[i] = nbr_id[i] >= 0 ? exp(beta * (weighted ? nbr_w[i] : 1.0)) : 1.0;
}

int launch_nbr_g(const int32_t *nbr_id, const double *nbr_w, double *nbr_g, int64_t count, double beta, int weighted,
                 cudaStream_t s) {
    if (count <= 0) return PHMRF_OK;
    const int64_t blocks = (count + 255) / 256;
    nbr_g_kernel<<<(int)(blocks < 2368 ? blocks : 2368), 256, 0, s>>>(nbr_id, nbr_w, nbr_g, count, beta, weighted);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

int launch_estep(const EstepArgs &a, int sm_count, cudaStream_t s) {
    if (a.n == 0) {
        PHMRF_CUDA(cudaMemsetAsync(a.stats_out, 0, sizeof(double) * (a.K * (1 + a.D + a.D * a.D) + 3), s));
        return PHMRF_OK;
    }
    switch (a.D) {
#define PHMRF_CASE(DD) \
    case DD:           \
        return launch_estep_d<DD>(a, sm_count, s);
        PHMRF_CASE(1) PHMRF_CASE(2) PHMRF_CASE(3) PHMRF_CASE(4) PHMRF_CASE(5) PHMRF_CASE(6)
        PHMRF_CASE(7) PHMRF_CASE(8) PHMRF_CASE(9) PHMRF_CASE(10) PHMRF_CASE(11) PHMRF_CASE(12)
#undef PHMRF_CASE
    }
    set_error("n_features outside [1,12]");
    return PHMRF_E_UNSUPPORTED;
}

}  // namespace phmrf
