// Per-node summary of the posterior over the K states (phmrf_posterior_summary): what the E-step's
// soft-max (phylo_hmrf.py:334-355) knows about each node, reduced to four numbers so that it can be kept
// for the whole fit instead of the dense [n, K] posterior.
//
// One lane per owned node and one pass over the states:
//   pp_k = sum_{j in N(i)} V[l_j, k] * w_ij   (w_ij = 1 unless estimate_type == 3; an isolated node takes
//          pp_k = V[l_i, k] unweighted, phylo_hmrf.py:421-423); Potts V: pp_k = wtot - S_k with beta folded
//          into the weights, S_k the weight of the neighbours labelled k, as phase B computes it
//   a_k  = logp_k - pp_k, m = max_k a_k, Z = sum_k exp(a_k - m)
//   map_state = first arg-max, map_prob = 1 / Z, label_prob = exp(a_{l_i} - m) / Z,
//   entropy = log Z - sum_k exp(a_k - m) (a_k - m) / Z
// m, Z and the entropy sum are kept online (rescaled when the maximum moves), so that any K takes one pass.
// The neighbour gather mirrors the general phase-B kernel for explicit slots and the pipeline kernel for
// grid-built regions; it is not shared with either: both fuse it with their own shared-memory or register
// layouts, and this pass only runs when a caller asks for it.
#include "estep_common.cuh"

namespace phmrf {

using namespace estep;

namespace {

constexpr int kSumThreads = 256;

// node id -> (row x, offset c in the row, row length L) in the reference's node order (utility.py:2310-2317):
// kind 1 the upper triangle of n2 bins (row x holds columns x..n2-1), kind 0 the n1 x n2 rectangle.  The same
// closed form as grid_locate of the pipeline kernel, whose header is private to its own translation units.
__device__ __forceinline__ void grid_row_of(int kind, long long n2, long long gid, int &x, int &c, int &L) {
    if (kind == 0) {
        const long long xx = gid / n2;
        x = (int)xx;
        c = (int)(gid - xx * n2);
        L = (int)n2;
        return;
    }
    const double bf = (double)n2 + 0.5;
    long long xx = (long long)(bf - sqrt(bf * bf - 2.0 * (double)gid));
    xx = xx < 0 ? 0 : (xx > n2 - 1 ? n2 - 1 : xx);
    auto start = [&](long long r) { return r * n2 - (r * (r - 1)) / 2; };
    while (xx > 0 && start(xx) > gid) --xx;
    while (xx < n2 - 1 && start(xx + 1) <= gid) ++xx;
    x = (int)xx;
    c = (int)(gid - start(xx));
    L = (int)(n2 - xx);
}

// adds one state's term to the online soft-max (m, Z, T): Z = sum exp(a_k - m), T = sum exp(a_k - m)(a_k - m); one
// exp per state, exp(-|a - m|) serving both the new term and the rescale when the maximum moves
__device__ __forceinline__ void online_add(double av, int k, double &m, double &Z, double &T, int &arg) {
    const double d = av - m;
    const double e = exp(-fabs(d));
    if (d > 0.0) {
        T = e * (T - d * Z);
        Z = e * Z + 1.0;
        m = av;
        arg = k;
    } else {
        Z += e;
        T += e > 0.0 ? e * d : 0.0;
    }
}

template <bool GRID>
__global__ void __launch_bounds__(kSumThreads) posterior_summary_kernel(EstepArgs a, double *__restrict__ out_d,
                                                                        int32_t *__restrict__ out_state) {
    const int64_t n = a.n, ld = a.ld;
    const int K = a.K, KP = logp_rows(K);
    const bool weighted = a.estimate_type == 3;
    const double beta = a.beta;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t iw = a.own_offset + i;
        const int li = a.labels[iw];
        // neighbours: label and weight as pp counts it (w, or 1), up to 8 in registers
        int lab[kFastSlots];
        double wt[kFastSlots];
        int W = GRID ? kFastSlots : a.W;
        if constexpr (GRID) {
            int x, c, L;
            grid_row_of(a.grid_kind, a.grid_n2, a.own_start_gid + i, x, c, L);
            const bool tri = a.grid_kind != 0;
            const int rows = (int)a.grid_rows;
            const bool nn8 = a.grid_nn == 8;
            const bool up = x > 0, down = x < rows - 1, left = c > 0, right = c < L - 1;
            const int dN = tri ? -L : -(int)a.grid_n2, dS = tri ? L - 1 : (int)a.grid_n2;
            // NW, N, NE, W, E, SW, S, SE; the weight lives with the edge's forward end (slot 0 right, 1 lower
            // left, 2 lower, 3 lower right), so a backward neighbour's weight is read from that neighbour
            const bool v[kFastSlots] = {nn8 && up && (tri || left), up, nn8 && up && right, left, right,
                                        nn8 && down && (tri ? c >= 2 : left), down && (tri ? c >= 1 : true),
                                        nn8 && (tri ? right : (down && right))};
            const int dl[kFastSlots] = {dN - 1, dN, dN + 1, -1, 1, dS - 1, dS, dS + 1};
            const int fs[kFastSlots] = {3, 2, 1, 0, 0, 1, 2, 3};
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                lab[s] = v[s] ? a.labels[iw + dl[s]] : -1;
                wt[s] = v[s] ? (weighted ? a.fwd_wg[fs[s] * a.ldw + iw + (s < 4 ? dl[s] : 0)].x : 1.0) : 0.0;
            }
        } else {
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) {
                const int j = s < W ? a.nbr_id[s * ld + i] : -1;
                lab[s] = j >= 0 ? a.labels[j] : -1;
                wt[s] = j >= 0 ? (weighted ? a.nbr_w[s * ld + i] : 1.0) : 0.0;
            }
        }
        // slots beyond the eighth (explicit graphs of higher degree) are read again for every state
        auto extra = [&](int s, int &l, double &w) {
            const int j = a.nbr_id[s * ld + i];
            l = j >= 0 ? a.labels[j] : -1;
            w = j >= 0 ? (weighted ? a.nbr_w[s * ld + i] : 1.0) : 0.0;
        };
        bool any = false;
#pragma unroll
        for (int s = 0; s < kFastSlots; ++s) any |= lab[s] >= 0;
        for (int s = kFastSlots; s < W && !any; ++s) any = a.nbr_id[s * ld + i] >= 0;
        if (!any) {  // isolated node: pp = V[l_i, :], unweighted
            lab[0] = li;
            wt[0] = 1.0;
            W = 1;
        }
        double wtot = 0.0;  // Potts: beta * sum of the weights
        if (a.potts) {
#pragma unroll
            for (int s = 0; s < kFastSlots; ++s) wtot += beta * wt[s];
            for (int s = kFastSlots; s < W; ++s) {
                int l;
                double w;
                extra(s, l, w);
                wtot += beta * w;
            }
        }
        // states in chunks of 8: the chunk's log-likelihood loads are issued together
        double m = -INFINITY, Z = 0.0, T = 0.0, a_li = 0.0;
        int arg = 0;
        for (int k0 = 0; k0 < K; k0 += 8) {
            double lp[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) lp[u] = k0 + u < K ? a.logp[lp_index(k0 + u, i, KP)] : 0.0;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int k = k0 + u;
                if (k >= K) break;
                double pp = 0.0;
                if (a.potts) {
                    double S = 0.0;
#pragma unroll
                    for (int s = 0; s < kFastSlots; ++s) S += lab[s] == k ? beta * wt[s] : 0.0;
                    for (int s = kFastSlots; s < W; ++s) {
                        int l;
                        double w;
                        extra(s, l, w);
                        S += l == k ? beta * w : 0.0;
                    }
                    pp = wtot - S;
                } else {
#pragma unroll
                    for (int s = 0; s < kFastSlots; ++s)
                        if (lab[s] >= 0) pp += a.V[lab[s] * K + k] * wt[s];
                    for (int s = kFastSlots; s < W; ++s) {
                        int l;
                        double w;
                        extra(s, l, w);
                        if (l >= 0) pp += a.V[l * K + k] * w;
                    }
                }
                const double av = lp[u] - pp;
                if (k == li) a_li = av;
                if (k == 0) {
                    m = av;
                    Z = 1.0;
                } else {
                    online_add(av, k, m, Z, T, arg);
                }
            }
        }
        const double inv = 1.0 / Z;
        out_d[i] = inv;                            // map_prob
        out_d[n + i] = exp(a_li - m) * inv;        // label_prob
        out_d[2 * n + i] = log(Z) - T * inv;       // entropy
        out_state[i] = arg;
    }
}

}  // namespace

int launch_posterior_summary(const EstepArgs &a, double *out_d, int32_t *out_state, int sm_count, cudaStream_t s) {
    if (a.n == 0) return PHMRF_OK;
    const int64_t want = (a.n + kSumThreads - 1) / kSumThreads, cap = (int64_t)sm_count * 8;
    const int grid = (int)(want < cap ? want : cap);
    if (a.fwd_wg != nullptr)
        posterior_summary_kernel<true><<<grid, kSumThreads, 0, s>>>(a, out_d, out_state);
    else
        posterior_summary_kernel<false><<<grid, kSumThreads, 0, s>>>(a, out_d, out_state);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

}  // namespace phmrf
