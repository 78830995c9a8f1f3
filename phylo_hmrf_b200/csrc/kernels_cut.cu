// Alpha-beta swap of csrc/gco.cpp on the device (phmrf_graph_cut_swap, phmrf_region_graph_cut).
//
//  * moves   the label pairs (a, b) in GCO's order: a ascending, b from K-1 down to a+1; cycles and
//            stopping rule as GeneralGraphCut::cycles.
//  * move    the sites labelled a or b are compacted; each builds its own terminal capacity and the
//            capacities of its arcs to the other active sites from the move's binary energy, in the
//            form E(x,y) = A + (C-A) x + (D-C) y + (B+C-A-D) (1-x) y for a pair (x the larger site).
//            That graph represents the same energy as the host's construction (both are exact
//            representations up to a constant), so the cut below is the host's cut.
//  * cut     synchronous push-relabel, phase 1 only, over the compacted sites.  Heights are fixed
//            during a push sweep, so at most one arc of a pair is admissible and only the pushing
//            site touches the pair's residual capacities; incoming excess goes to a separate buffer
//            that the relabel sweep merges.  Global relabels (distance to the sink over residual arcs,
//            relaxed to the fixed point) run at the start and every few batches.  When no site with
//            excess has a finite height, one more relabel gives the sites that reach the sink in the
//            residual graph: those take b.  That set (the smallest sink side of all minimum cuts)
//            depends on the energy alone, so the labels equal the host's move for move.
//  * bounds  every kernel is a grid-stride pass over the sites or arcs; the host drives the sweeps and
//            reads a few control words through host-mapped memory between batches.
#include <climits>

#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace phmrf {

namespace {

constexpr long long kMaxTerm = 10000000;  // GCO_MAX_ENERGYTERM
constexpr int kInf = 0x3fffffff;          // height of a site that cannot reach the sink
constexpr int kThreads = 256;
constexpr int kMaxBlocks = 148 * 8;
constexpr int kSweepsPerCheck = 16;       // push + relabel sweeps between two reads of the active count
constexpr int kBatchesPerRelabel = 4;     // global relabel after this many batches
constexpr int kPassesPerCheck = 8;        // relaxation passes of a global relabel between two reads

// control words (device memory; published to the host-mapped copy)
enum { kCtlNAct = 0, kCtlErr = 1, kCtlEnergy = 2, kCtlMinW = 3, kCtlActive = 4 /* 2 words */,
       kCtlChanged = 6 /* 2 words */, kCtlWords = 8 };

int grid_for(int64_t count) {
    const int64_t b = (count + kThreads - 1) / kThreads;
    return (int)(b < 1 ? 1 : (b > kMaxBlocks ? kMaxBlocks : b));
}

// every launch of this file: grid-stride kernels over `count` items on stream `st`
#define LAUNCH(kernel, count, ...)                                              \
    do {                                                                        \
        kernel<<<grid_for(count), kThreads, 0, st>>>(__VA_ARGS__);              \
        count_launch();                                                         \
        PHMRF_CUDA(cudaGetLastError());                                         \
    } while (0)

__device__ __forceinline__ void add_ll(long long *p, long long v) {
    atomicAdd(reinterpret_cast<unsigned long long *>(p), (unsigned long long)v);
}

__device__ __forceinline__ long long warp_sum(long long v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------- graph (CSR with edge index and reverse slot)
__global__ void edge_degree_kernel(const long long *ids, int64_t E, unsigned long long *deg) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
        atomicAdd(&deg[ids[2 * e]], 1ull);
        atomicAdd(&deg[ids[2 * e + 1]], 1ull);
    }
}

__global__ void edge_fill_kernel(const long long *ids, int64_t E, unsigned long long *cursor, long long *nbr,
                                 long long *eid, long long *rev) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
        const long long a = ids[2 * e], b = ids[2 * e + 1];
        const long long ka = (long long)atomicAdd(&cursor[a], 1ull), kb = (long long)atomicAdd(&cursor[b], 1ull);
        nbr[ka] = b; eid[ka] = e; rev[ka] = kb;
        nbr[kb] = a; eid[kb] = e; rev[kb] = ka;
    }
}

// ELL slots [W][ld] (-1 = empty): degree and forward degree (neighbours with a larger id) per site
__global__ void ell_degree_kernel(const int32_t *nbr_id, int W, int64_t ld, int64_t n, long long *deg,
                                  long long *fdeg) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        long long d = 0, f = 0;
        for (int s = 0; s < W; ++s) {
            const int32_t j = nbr_id[(int64_t)s * ld + i];
            d += j >= 0;
            f += j > i;
        }
        deg[i] = d;
        fdeg[i] = f;
    }
}

// With the edge list sorted by (id1, id2), edge (lo, hi) is number fstart[lo] + (lo's forward neighbours below
// hi) + (copies of the same edge before it, in slot order, which is edge order).  pos[e] / pos[E + e] record the
// slot of the lower / upper end.
__global__ void ell_fill_kernel(const int32_t *nbr_id, int W, int64_t ld, int64_t n, int64_t E, const long long *start,
                                const long long *fstart, long long *nbr, long long *eid, long long *pos) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        long long k = start[i];
        for (int s = 0; s < W; ++s) {
            const int64_t j = nbr_id[(int64_t)s * ld + i];
            if (j < 0) continue;
            const int64_t lo = j < i ? j : i, hi = j < i ? i : j;
            long long r = 0;
            for (int q = 0; q < W; ++q) {
                const int64_t t = nbr_id[(int64_t)q * ld + lo];
                r += t > lo && t < hi;
            }
            for (int q = 0; q < s; ++q) r += nbr_id[(int64_t)q * ld + i] == j;
            const long long e = fstart[lo] + r;
            pos[(j > i ? 0 : E) + e] = k;
            nbr[k] = j;
            eid[k] = e;
            ++k;
        }
    }
}

__global__ void ell_rev_kernel(int64_t n, int64_t E, const long long *start, const long long *nbr, const long long *eid,
                               const long long *pos, long long *rev) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        for (long long k = start[i]; k < start[i + 1]; ++k) rev[k] = nbr[k] > i ? pos[E + eid[k]] : pos[eid[k]];
}

__global__ void gather_weights_kernel(int64_t slots, const long long *eid, const int32_t *w_edge, int32_t *wslot,
                                      long long *ctl) {
    long long wmin = LLONG_MAX;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < slots; k += (int64_t)gridDim.x * blockDim.x) {
        const int32_t w = w_edge[eid[k]];
        wslot[k] = w;
        wmin = w < wmin ? w : wmin;
    }
    if (wmin < 0) atomicMin(&ctl[kCtlMinW], wmin);
}

__global__ void fill_ll_kernel(long long *p, int64_t count, long long v) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
        p[i] = v;
}

// ---------------------------------------------------------------- energy and moves
// E(l) = sum_s D[s][l_s] + sum_{edges t<s} w * V[l_s][l_t], added into ctl[kCtlEnergy]
__global__ void energy_kernel(int64_t n, int K, const int32_t *unary, const long long *start, const long long *nbr,
                              const int32_t *wslot, const int32_t *V, const int32_t *labels, long long *ctl) {
    long long acc = 0;
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
        const int ls = labels[s];
        acc += unary[s * K + ls];
        for (long long k = start[s]; k < start[s + 1]; ++k) {
            const long long t = nbr[k];
            if (t < s) acc += (long long)wslot[k] * V[ls * K + labels[t]];
        }
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0 && acc != 0) add_ll(&ctl[kCtlEnergy], acc);
}

__global__ void compact_kernel(int64_t n, const int32_t *labels, int a, int b, long long *act, long long *var,
                               long long *ctl) {
    const int lane = threadIdx.x & 31;
    for (int64_t base = blockIdx.x * (int64_t)blockDim.x; base < n; base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = base + threadIdx.x;
        bool in = false;
        if (s < n) {
            const int l = labels[s];
            in = l == a || l == b;
        }
        const unsigned m = __ballot_sync(0xffffffffu, in);
        long long first = 0;
        if (lane == 0 && m) first = (long long)atomicAdd(reinterpret_cast<unsigned long long *>(&ctl[kCtlNAct]),
                                                         (unsigned long long)__popc(m));
        first = __shfl_sync(0xffffffffu, first, 0);
        if (in) {
            const long long i = first + __popc(m & ((1u << lane) - 1u));
            act[i] = s;
            var[s] = i;
        }
    }
}

// Terminal and arc capacities of the move (a: x = 0, b: x = 1); the first term above GCO_MAX_ENERGYTERM in
// the host's order of checks lands in ctl[kCtlErr] as 2*site + (0 data, 1 smooth).
__global__ void setup_kernel(int K, const int32_t *unary, const long long *start, const long long *nbr,
                             const int32_t *wslot, const int32_t *V, const int32_t *labels, const long long *act, int a,
                             int b, long long *excess, long long *tcap, long long *inflow, long long *rcap,
                             long long *ctl) {
    const long long n_act = ctl[kCtlNAct];
    const long long Vaa = V[a * K + a], Vab = V[a * K + b], Vba = V[b * K + a], Vbb = V[b * K + b];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_act; i += (int64_t)gridDim.x * blockDim.x) {
        const long long s = act[i];
        const long long e0 = unary[s * K + a], e1 = unary[s * K + b];
        long long code = (e0 > kMaxTerm || e1 > kMaxTerm) ? 2 * s : LLONG_MAX;
        long long tr = e1 - e0;  // > 0: capacity from the source, < 0: to the sink
        for (long long k = start[s]; k < start[s + 1]; ++k) {
            const long long t = nbr[k];
            const long long w = wslot[k];
            const int lt = labels[t];
            if (lt == a || lt == b) {
                // V indexed [larger site][smaller site]; x = the larger site
                const long long A = w * Vaa, B = w * Vab, C = w * Vba, D = w * Vbb;
                if ((A > kMaxTerm || B > kMaxTerm || C > kMaxTerm || D > kMaxTerm) && 2 * (t > s ? t : s) + 1 < code)
                    code = 2 * (t > s ? t : s) + 1;
                if (t < s) {
                    tr += C - A;
                    rcap[k] = B + C - A - D;
                } else {
                    tr += D - C;
                    rcap[k] = 0;
                }
            } else {
                const long long e0n = w * V[a * K + lt], e1n = w * V[b * K + lt];
                if ((e0n > kMaxTerm || e1n > kMaxTerm) && 2 * s + 1 < code) code = 2 * s + 1;
                tr += e1n - e0n;
                rcap[k] = 0;
            }
        }
        excess[i] = tr > 0 ? tr : 0;
        tcap[i] = tr < 0 ? -tr : 0;
        inflow[i] = 0;
        if (code != LLONG_MAX) atomicMin(&ctl[kCtlErr], code);
    }
}

__global__ void height_init_kernel(int64_t n_act, const long long *tcap, int *h) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_act; i += (int64_t)gridDim.x * blockDim.x)
        h[i] = tcap[i] > 0 ? 1 : kInf;
}

// One relaxation pass of the distance to the sink over residual arcs; counts the sites it lowered in
// ctl[kCtlChanged + parity] and clears the other parity's word for the next pass.  Heights only decrease and
// every value written is one more than a neighbour's, so the fixed point is the exact distance.
__global__ void relax_kernel(int64_t n_act, const long long *act, const long long *start, const long long *nbr,
                             const long long *var, const long long *rcap, int *h, long long *ctl, int parity) {
    if (blockIdx.x == 0 && threadIdx.x == 0) ctl[kCtlChanged + (parity ^ 1)] = 0;
    long long changed = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_act; i += (int64_t)gridDim.x * blockDim.x) {
        const int hi = h[i];
        if (hi == 1) continue;
        const long long s = act[i];
        int m = hi;
        for (long long k = start[s]; k < start[s + 1]; ++k)
            if (rcap[k] > 0) {
                const int hj = ((volatile int *)h)[var[nbr[k]]];
                if (hj + 1 < m) m = hj + 1;
            }
        if (m < hi) {
            h[i] = m;
            ++changed;
        }
    }
    changed = warp_sum(changed);
    if ((threadIdx.x & 31) == 0 && changed) add_ll(&ctl[kCtlChanged + parity], changed);
}

// Push sweep: heights are read only, so an admissible arc's reverse is not admissible and only this site
// changes the pair's residual capacities; the neighbour's share goes to inflow.
__global__ void push_kernel(int64_t n_act, const long long *act, const long long *start, const long long *nbr,
                            const long long *var, const long long *rev, long long *rcap, const int *h,
                            long long *excess, long long *tcap, long long *inflow) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_act; i += (int64_t)gridDim.x * blockDim.x) {
        long long e = excess[i];
        if (e <= 0) continue;
        const int hi = h[i];
        if (hi >= kInf) continue;
        if (hi == 1) {
            const long long tc = tcap[i];
            if (tc > 0) {
                const long long d = e < tc ? e : tc;
                tcap[i] = tc - d;
                e -= d;
            }
        }
        if (e > 0) {
            const long long s = act[i];
            for (long long k = start[s]; k < start[s + 1] && e > 0; ++k) {
                const long long rc = rcap[k];
                if (rc <= 0) continue;
                const long long j = var[nbr[k]];
                if (h[j] != hi - 1) continue;
                const long long d = e < rc ? e : rc;
                rcap[k] = rc - d;
                rcap[rev[k]] += d;
                add_ll(&inflow[j], d);
                e -= d;
            }
        }
        excess[i] = e;
    }
}

// Relabel sweep: merge the inflow, lift every site with excess to one above its lowest residual neighbour
// (a height above n_act cannot reach the sink), count the sites that still hold excess at a finite height.
__global__ void relabel_kernel(int64_t n_act, const long long *act, const long long *start, const long long *nbr,
                               const long long *var, const long long *rcap, int *h, long long *excess,
                               const long long *tcap, long long *inflow, long long *ctl, int parity) {
    if (blockIdx.x == 0 && threadIdx.x == 0) ctl[kCtlActive + (parity ^ 1)] = 0;
    long long active = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_act; i += (int64_t)gridDim.x * blockDim.x) {
        long long e = excess[i];
        const long long in = inflow[i];
        if (in) {
            e += in;
            inflow[i] = 0;
            excess[i] = e;
        }
        if (e <= 0 || h[i] >= kInf) continue;
        long long m = kInf;
        if (tcap[i] > 0) {
            m = 0;
        } else {
            const long long s = act[i];
            for (long long k = start[s]; k < start[s + 1]; ++k)
                if (rcap[k] > 0) {
                    const int hj = ((volatile int *)h)[var[nbr[k]]];
                    if (hj < m) m = hj;
                }
        }
        const int nh = (m >= kInf || m + 1 > n_act) ? kInf : (int)(m + 1);
        h[i] = nh;
        active += nh < kInf;
    }
    active = warp_sum(active);
    if ((threadIdx.x & 31) == 0 && active) add_ll(&ctl[kCtlActive + parity], active);
}

__global__ void apply_kernel(int64_t n_act, const long long *act, const int *h, int a, int b, int32_t *labels,
                             long long *var) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_act; i += (int64_t)gridDim.x * blockDim.x) {
        const long long s = act[i];
        labels[s] = h[i] < kInf ? b : a;
        var[s] = -1;
    }
}

int exclusive_scan(const long long *in, long long *out, int64_t count, cudaStream_t st) {
    size_t bytes = 0;
    PHMRF_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, count, st));
    DevBuf<unsigned char> tmp;
    int rc = tmp.alloc((int64_t)bytes);
    if (rc) return rc;
    PHMRF_CUDA(cub::DeviceScan::ExclusiveSum(tmp.get(), bytes, in, out, count, st));
    PHMRF_CUDA(cudaStreamSynchronize(st));
    count_launch();
    return PHMRF_OK;
}

// the control words as the host sees them after the stream drains
int read_ctl(SwapScratch &s, cudaStream_t st, long long *out) {
    int rc = launch_publish(s.map.dev, s.ctl, kCtlWords, false, st);
    if (rc) return rc;
    PHMRF_CUDA(cudaStreamSynchronize(st));
    for (int w = 0; w < kCtlWords; ++w) out[w] = (long long)s.map.host[w];
    return PHMRF_OK;
}

int energy(SwapScratch &s, const int32_t *unary, const int32_t *labels, cudaStream_t st, long long *en) {
    PHMRF_CUDA(cudaMemsetAsync(s.ctl + kCtlEnergy, 0, sizeof(long long), st));
    LAUNCH(energy_kernel, s.n, s.n, s.K, unary, s.start, s.nbr, s.wslot, s.V, labels, s.ctl);
    long long c[kCtlWords];
    int rc = read_ctl(s, st, c);
    if (rc) return rc;
    *en = c[kCtlEnergy];
    return PHMRF_OK;
}

// exact distances to the sink over residual arcs (kInf: cannot reach it)
int global_relabel(SwapScratch &s, int64_t n_act, cudaStream_t st) {
    LAUNCH(height_init_kernel, n_act, n_act, s.tcap, s.h);
    PHMRF_CUDA(cudaMemsetAsync(s.ctl + kCtlChanged, 0, 2 * sizeof(long long), st));
    // a distance is at most n_act, so n_act + 1 passes reach the fixed point
    for (int64_t pass = 0; pass <= n_act + 1;) {
        for (int q = 0; q < kPassesPerCheck; ++q, ++pass)
            LAUNCH(relax_kernel, n_act, n_act, s.act, s.start, s.nbr, s.var, s.rcap, s.h, s.ctl, (int)(pass & 1));
        long long c[kCtlWords];
        int rc = read_ctl(s, st, c);
        if (rc) return rc;
        if (c[kCtlChanged + (int)((pass - 1) & 1)] == 0) return PHMRF_OK;
    }
    set_error("GCO (device swap): distance labelling did not converge");
    return PHMRF_E_STATE;
}

int swap_move(SwapScratch &s, const int32_t *unary, int32_t *labels, int a, int b, cudaStream_t st) {
    PHMRF_CUDA(cudaMemsetAsync(s.ctl + kCtlNAct, 0, sizeof(long long), st));
    PHMRF_CUDA(cudaMemsetAsync(s.ctl + kCtlActive, 0, 4 * sizeof(long long), st));
    LAUNCH(compact_kernel, s.n, s.n, labels, a, b, s.act, s.var, s.ctl);
    LAUNCH(setup_kernel, s.n, s.K, unary, s.start, s.nbr, s.wslot, s.V, labels, s.act, a, b, s.excess, s.tcap,
           s.inflow, s.rcap, s.ctl);
    long long c[kCtlWords];
    int rc = read_ctl(s, st, c);
    if (rc) return rc;
    if (c[kCtlErr] != LLONG_MAX) {
        set_error((c[kCtlErr] & 1) ? "GCO: smooth cost term larger than GCO_MAX_ENERGYTERM (1e7): danger of integer overflow"
                                   : "GCO: data cost term larger than GCO_MAX_ENERGYTERM (1e7): danger of integer overflow");
        return PHMRF_E_INVALID;
    }
    const int64_t n_act = c[kCtlNAct];
    if (n_act == 0) return PHMRF_OK;
    if ((rc = global_relabel(s, n_act, st)) != PHMRF_OK) return rc;
    // phase 1 of push-relabel needs O(n^2) sweeps at most; the bound only keeps a defect from looping
    const double cap = 4.0 * ((double)n_act + 2.0) * ((double)n_act + 2.0) + 1e6;
    int64_t sweep = 0;
    for (int batch = 1;; ++batch) {
        for (int q = 0; q < kSweepsPerCheck; ++q, ++sweep) {
            LAUNCH(push_kernel, n_act, n_act, s.act, s.start, s.nbr, s.var, s.rev, s.rcap, s.h, s.excess, s.tcap,
                   s.inflow);
            LAUNCH(relabel_kernel, n_act, n_act, s.act, s.start, s.nbr, s.var, s.rcap, s.h, s.excess, s.tcap, s.inflow,
                   s.ctl, (int)(sweep & 1));
        }
        if ((rc = read_ctl(s, st, c)) != PHMRF_OK) return rc;
        if (c[kCtlActive + (int)((sweep - 1) & 1)] == 0) break;
        if ((double)sweep > cap) {
            set_error("GCO (device swap): push-relabel did not converge");
            return PHMRF_E_STATE;
        }
        if (batch % kBatchesPerRelabel == 0 && (rc = global_relabel(s, n_act, st)) != PHMRF_OK) return rc;
    }
    // the sites that reach the sink in the residual graph of the maximum preflow take b
    if ((rc = global_relabel(s, n_act, st)) != PHMRF_OK) return rc;
    LAUNCH(apply_kernel, n_act, n_act, s.act, s.h, a, b, labels, s.var);
    return PHMRF_OK;
}

}  // namespace

int swap_scratch_alloc(SwapScratch &s, int64_t n, int64_t E, int K) {
    s.n = n;
    s.E = E;
    s.K = K;
    const int64_t slots = 2 * E;
    int64_t *b = &s.bytes;
    int rc;
    if ((rc = s.start.alloc(n + 1, b)) || (rc = s.nbr.alloc(slots, b)) || (rc = s.eid.alloc(slots, b)) ||
        (rc = s.rev.alloc(slots, b)) || (rc = s.rcap.alloc(slots, b)) || (rc = s.wslot.alloc(slots, b)) ||
        (rc = s.act.alloc(n, b)) || (rc = s.var.alloc(n + 1, b)) || (rc = s.excess.alloc(n + 1, b)) ||
        (rc = s.inflow.alloc(n, b)) || (rc = s.tcap.alloc(n, b)) || (rc = s.h.alloc(n, b)) ||
        (rc = s.V.alloc((int64_t)K * K, b)) || (rc = s.ctl.alloc(kCtlWords, b)))
        return rc;
    return s.map.alloc(kCtlWords);
}

int swap_graph_from_edges(SwapScratch &s, const long long *edge_ids, cudaStream_t st) {
    unsigned long long *deg = reinterpret_cast<unsigned long long *>(s.excess.get());  // [n+1] counts, then cursors
    PHMRF_CUDA(cudaMemsetAsync(deg, 0, sizeof(long long) * (s.n + 1), st));
    if (s.E > 0) LAUNCH(edge_degree_kernel, s.E, edge_ids, s.E, deg);
    int rc = exclusive_scan(s.excess, s.start, s.n + 1, st);
    if (rc) return rc;
    PHMRF_CUDA(cudaMemcpyAsync(deg, s.start, sizeof(long long) * (s.n + 1), cudaMemcpyDeviceToDevice, st));
    if (s.E > 0) LAUNCH(edge_fill_kernel, s.E, edge_ids, s.E, deg, s.nbr, s.eid, s.rev);
    LAUNCH(fill_ll_kernel, s.n, s.var, s.n, -1ll);
    return PHMRF_OK;
}

int swap_graph_from_ell(SwapScratch &s, const int32_t *nbr_id, int W, int64_t ld, cudaStream_t st) {
    long long *deg = s.excess, *fdeg = s.var, *fstart = s.act;  // [n+1] temporaries ([n] for act: fstart[n] unused)
    PHMRF_CUDA(cudaMemsetAsync(deg, 0, sizeof(long long) * (s.n + 1), st));
    PHMRF_CUDA(cudaMemsetAsync(fdeg, 0, sizeof(long long) * (s.n + 1), st));
    if (W > 0) LAUNCH(ell_degree_kernel, s.n, nbr_id, W, ld, s.n, deg, fdeg);
    int rc = exclusive_scan(deg, s.start, s.n + 1, st);
    if (rc) return rc;
    if ((rc = exclusive_scan(fdeg, fstart, s.n, st))) return rc;
    if (W > 0 && s.E > 0) {
        LAUNCH(ell_fill_kernel, s.n, nbr_id, W, ld, s.n, s.E, s.start, fstart, s.nbr, s.eid, s.rcap);
        LAUNCH(ell_rev_kernel, s.n, s.n, s.E, s.start, s.nbr, s.eid, s.rcap, s.rev);
    }
    LAUNCH(fill_ll_kernel, s.n, s.var, s.n, -1ll);
    return PHMRF_OK;
}

int swap_run(SwapScratch &s, const int32_t *unary, const int32_t *w_edge, const int32_t *V_host, int32_t *labels,
             int n_iter, long long *energy_out, long long *energy_before_out, cudaStream_t st) {
    const int K = s.K;
    for (int a = 0; a < K; ++a)
        for (int b = 0; b < K; ++b)
            if (a != b && (long long)V_host[a * K + b] + V_host[b * K + a] < (long long)V_host[a * K + a] + V_host[b * K + b]) {
                set_error("GCO (device swap): smooth costs with V[a][b] + V[b][a] < V[a][a] + V[b][b] make a "
                          "non-submodular move; only the host cut runs them");
                return PHMRF_E_UNSUPPORTED;
            }
    PHMRF_CUDA(cudaMemcpyAsync(s.V, V_host, sizeof(int32_t) * K * K, cudaMemcpyHostToDevice, st));
    const long long init[kCtlWords] = {0, LLONG_MAX, 0, LLONG_MAX, 0, 0, 0, 0};
    PHMRF_CUDA(cudaMemcpyAsync(s.ctl, init, sizeof(init), cudaMemcpyHostToDevice, st));
    if (s.E > 0) LAUNCH(gather_weights_kernel, 2 * s.E, 2 * s.E, s.eid, w_edge, s.wslot, s.ctl);
    long long c[kCtlWords];
    int rc = read_ctl(s, st, c);
    if (rc) return rc;
    if (c[kCtlMinW] < 0) {
        set_error("GCO (device swap): negative edge weights make non-submodular moves; only the host cut runs them");
        return PHMRF_E_UNSUPPORTED;
    }
    long long en = 0;
    if ((rc = energy(s, unary, labels, st, &en)) != PHMRF_OK) return rc;
    if (energy_before_out) *energy_before_out = en;
    const long long n_max = n_iter == -1 ? LLONG_MAX : n_iter;
    long long old = en + 1;
    for (long long cyc = 1; old > en && cyc <= n_max; ++cyc) {
        old = en;
        for (int a = 0; a < K; ++a)
            for (int b = K - 1; b > a; --b)
                if ((rc = swap_move(s, unary, labels, a, b, st)) != PHMRF_OK) return rc;
        if ((rc = energy(s, unary, labels, st, &en)) != PHMRF_OK) return rc;
    }
    if (energy_out) *energy_out = en;
    return PHMRF_OK;
}

}  // namespace phmrf
