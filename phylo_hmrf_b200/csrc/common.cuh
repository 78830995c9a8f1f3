// Shared declarations between the host API (api.cu) and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <limits>
#include <string>

#include "../../include/phmrf.h"

namespace phmrf {

constexpr int kMinFeatures = 1;
constexpr int kMaxFeatures = 12;      // D is a template parameter of the kernels

void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);
void count_launch(int n = 1);

#define PHMRF_CUDA(expr)                                                       \
    do {                                                                       \
        cudaError_t _e = (expr);                                               \
        if (_e != cudaSuccess) return ::phmrf::cuda_fail(_e, #expr, __FILE__, __LINE__); \
    } while (0)

// The owners of the library's device and mapped memory: nothing else frees it.

// One cudaMalloc of T, freed by the destructor.  Converts to T * so that launch sites read as with a raw pointer.
template <typename T>
class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p_(o.p_) { o.p_ = nullptr; }
    ~DevBuf() {
        if (p_) cudaFree(p_);
    }
    // Frees what it holds and allocates `count` elements (at least one); adds their size to *bytes when given.
    int alloc(int64_t count, int64_t *bytes = nullptr) {
        if (p_) cudaFree(p_);
        p_ = nullptr;
        if (count <= 0) count = 1;
        PHMRF_CUDA(cudaMalloc((void **)&p_, sizeof(T) * (size_t)count));
        if (bytes) *bytes += (int64_t)sizeof(T) * count;
        return PHMRF_OK;
    }
    T *get() const { return p_; }
    operator T *() const { return p_; }

  private:
    T *p_ = nullptr;
};

// One pinned host block of 64-bit words mapped into the device (cudaHostAllocMapped | Portable): kernels store
// small results through `dev` (launch_publish) and the host reads them through `host` after a stream sync.
struct MappedBuf {
    unsigned long long *host = nullptr, *dev = nullptr;
    MappedBuf() = default;
    MappedBuf(const MappedBuf &) = delete;
    MappedBuf &operator=(const MappedBuf &) = delete;
    ~MappedBuf() {
        if (host) cudaFreeHost(host);
    }
    int alloc(size_t words) {
        PHMRF_CUDA(cudaHostAlloc((void **)&host, words * sizeof(unsigned long long),
                                 cudaHostAllocMapped | cudaHostAllocPortable));
        PHMRF_CUDA(cudaHostGetDevicePointer((void **)&dev, host, 0));
        return PHMRF_OK;
    }
};

// Per-state emission parameters as the kernels consume them (built on the host from the
// Cholesky factor): z = Wh*x - ch with Wh = sqrt(1/2)*L^-1 (lower triangular), ch = Wh*mu,
// and logp = -(hc + sum z^2) with hc = (d*ln(2pi) + logdet)/2.  Stored as the stream the
// emission kernel consumes: hc, then for each row i: ch_i, Wh_i0 .. Wh_ii.
__host__ __device__ constexpr int model_stride(int D) { return D * (D + 1) / 2 + D + 1; }
__host__ __device__ constexpr int n_stat_features(int D) { return 1 + D + D * (D + 1) / 2; }

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// Log-likelihood layout in HBM: tile-major, 32 nodes per tile, KP = logp_rows(K) state rows of
// 32 doubles per tile, the node column XOR-swizzled by the state row:
//   (k, i)  ->  ((i / 32) * KP + k) * 32 + ((i % 32) ^ ((k % 8) * 4))
// One tile (KP * 256 bytes) is contiguous, so phase B fetches it with ONE bulk copy
// (cp.async.bulk) straight into shared memory, where the swizzle makes both access patterns
// conflict free: a lane per node along a row (per-node warps) and the FP64 mma operand
// fragments (8 states x 4 nodes; tools/swizzle_check.py).  The XOR acts on multiples of 4,
// so groups of 4 consecutive nodes stay contiguous (the emission kernel's 128-bit stores).
__host__ __device__ __forceinline__ int64_t lp_index(int k, int64_t i, int KP) {
    return ((i >> 5) * KP + k) * 32 + ((i & 31) ^ ((k & 7) << 2));
}

// ---- phase A (kernels_a.cu) -----------------------------------------------------------
// X_aos [n,D] row-major -> X_soa [D][ld]
int launch_aos_to_soa(const double *X_aos, double *X_soa, int64_t n, int D, int64_t ld, cudaStream_t s);
// [K][ld] -> out [n,K] row-major (posteriors, pairwise potential)
int launch_soa_to_aos(const double *soa, double *aos, int64_t n, int K, int64_t ld, cudaStream_t s);
// log-likelihood: host order [n,K] row-major <-> the tiled device layout (lp_index)
int launch_logp_from_aos(const double *aos, double *logp, int64_t n, int K, cudaStream_t s);
int launch_logp_to_aos(const double *logp, double *aos, int64_t n, int K, cudaStream_t s);
// emission: logp[k][i] for i<n, block maxima of |logp| folded into *absmax_bits (uint64 bit
// pattern of a non-negative double, atomicMax).
int launch_emit(const double *X_soa, int64_t n, int64_t ld, int D, int K, const double *model_global,
                double *logp, unsigned long long *absmax_bits, int sm_count, cudaStream_t s);
// per-node maximum over the states (phase B's soft-max shift); the quantise kernel writes it
// on its way, this is the stand-alone form for a caller-supplied log-likelihood
int launch_rowmax(const double *logp, int64_t n, int K, double *rowmax, unsigned long long *absmax_bits,
                  cudaStream_t s);
int launch_check_labels(const int32_t *labels, int64_t n, int K, long long *first_bad, cudaStream_t s);
int launch_fill(double *p, double v, int64_t count, cudaStream_t s);
// Small results to the host without the copy engines: the kernel stores `count` 64-bit words (or,
// with src32, sign-extended 32-bit words) into a host-mapped pinned buffer.  A DMA read-back of a few
// bytes queues behind whatever bulk download another region has in flight (tens of milliseconds);
// stores from an SM do not.
int launch_publish(unsigned long long *dst_mapped, const void *src, int count, bool src32, cudaStream_t s);
// rows of the log-likelihood matrix: K rounded up to the 8-state tiles of the pipeline kernel.  The
// padding rows keep their values for the lifetime of a region: row K of an odd K holds kLogpPad (the
// pipeline evaluates states in pairs: exp(-inf - shift) lands on its exp's lower clamp, e^-704, for ANY
// shift -- a finite pad such as -1e6 outweighs the real states of a node whose log-likelihoods lie near or
// below it), the rows from the next even number on hold 0.0 -- the pipeline never evaluates them, and the
// bulk copy then drops a zero WEIGHT for them straight into the soft-max buffer the statistics product
// reads.  Every other reader of the log-likelihood stops at row K - 1.
__host__ __device__ inline int logp_rows(int K) { return (K + 7) / 8 * 8; }
constexpr double kLogpPad = -std::numeric_limits<double>::infinity();
int launch_logp_init(double *logp, int64_t ld, int K, cudaStream_t s);
// dwf = max(absmax_u, wmax*vmax) + 1e-10 unless dwf_in > 0; written to *dwf_dev.
int launch_dwf(const unsigned long long *absmax_bits, double wmax, double vmax, double dwf_in, double *dwf_dev,
               cudaStream_t s);
// unary_i32[i*K+k] = trunc(((-logp[k][i])/dwf)*uprec); boundary entries appended to blist;
// rowmax[i] = max_k logp[k][i]; and, in the same launch, w_i32[e] = trunc((w[e]/dwf)*wprec)
// for the E edge weights (edge_w == nullptr skips it).
int launch_quantise(const double *logp, int64_t n, int K, const double *dwf_dev, double tol, double uprec,
                    int32_t *unary, double *rowmax, long long *blist, long long bcap, unsigned long long *bcount,
                    const double *edge_w, int64_t E, double wprec, int32_t *w_i32, int sm_count, cudaStream_t s);
int launch_argmin_unary(const int32_t *unary, int64_t n, int K, int32_t *labels, cudaStream_t s);

// ---- phase B (kernels_b.cu) -----------------------------------------------------------
struct EstepArgs {
    const double *X_soa;      // [D][ld]
    const double *logp;       // tiled [n/32][KP][32], see lp_index
    const double *rowmax;     // [ld] max_k logp (pipeline kernel only)
    const int32_t *labels;    // [n_window]
    const int32_t *nbr_id;    // [W][ld] window-local neighbour id, -1 = none
    const double *nbr_w;      // [W][ld] edge weight per slot
    const double *V;          // [K][K] (general path only)
    double beta;              // Potts strength (fast path)
    int potts;
    int64_t n, ld, own_offset;
    int D, K, W, estimate_type;
    double *post_soa;         // nullable [K][ld]
    double *pp_soa;           // nullable [K][ld] pairwise potential (signature-parity output)
    double *partials;         // [sm_count][K*F + 3] per-CTA partial sums
    double *stats_out;        // [K*(1+D+D*D) + 3]
    int *flags;               // [1] device flag: bit 0 = the pipeline met an overflow, rerun on the general path
    int64_t own_start_gid;    // region-global node id of the first owned node (implicit-grid form, below)
    double s_bound;           // upper bound of any neighbour weight sum: beta * W * max|w|
    const double *nbr_g;      // [W][ld] exp(beta * w) per slot (1 for an empty slot); pipeline kernel only
    double exp_beta;          // exp(beta)
    // implicit-grid form (regions built by phmrf_region_create_grid): neighbours are fixed offsets
    // from the row geometry, each edge weight is stored once, with its forward end
    const double2 *fwd_wg;    // [4][ldw] per window node: {w, exp(beta*w)} of right, lower-left, lower, lower-right
    int64_t ldw;
    int grid_kind;            // 1 diagonal region (upper triangle), 0 rectangle, -1: explicit neighbour slots
    int grid_nn;              // 8 or 4
    int64_t grid_n2, grid_rows;
};
// g[s][i] = exp(beta * (weighted ? w[s][i] : 1)) for occupied slots, 1 otherwise (kernels_b.cu)
int launch_nbr_g(const int32_t *nbr_id, const double *nbr_w, double *nbr_g, int64_t count, double beta, int weighted,
                 cudaStream_t s);
// The general kernel (kernels_b.cu): any V, any degree, any K; n == 0 zero-fills the statistics.
int launch_estep(const EstepArgs &a, int sm_count, cudaStream_t s);
// The one decision between the two phase-B kernels: true when the warp-specialised bulk-copy pipeline
// (estep_bulk.cuh, kernels_b3*.cu) runs this E-step -- n > 0, no pp output, Potts V, 1..8 neighbour slots,
// |s_bound| < 100, K <= 40 and a kernel shape that fits the registers and shared memory.  The caller then
// fills nbr_g, or fwd_wg and grid_kind, and calls launch_estep_bulk, which returns PHMRF_E_UNSUPPORTED for
// any other shape.  The redo after an overflow flag always takes the general kernel.
bool estep_bulk_supported(const EstepArgs &a);
int launch_estep_bulk(const EstepArgs &a, int sm_count, cudaStream_t s);
// Fold per-block partials into stats_out (defined in kernels_b.cu).
int launch_estep_finalize(const double *partials, int n_blocks, int K, int D, double *stats_out, cudaStream_t s);
// Posterior summary of the owned nodes (kernels_summary.cu) from the inputs of the E-step: out_d [3][n] =
// map_prob | label_prob | entropy, out_state [n].  Reads the implicit grid when a.fwd_wg is set, else the
// neighbour slots.
int launch_posterior_summary(const EstepArgs &a, double *out_d, int32_t *out_state, int sm_count, cudaStream_t s);

// ---- SURVEY 8(f-1): region edge lists on the GPU (kernels_grid.cu) ----------------------
long long grid_edge_count(int kind, long long n1, long long n2, int nn);
int launch_grid_edges(const double *X_dev, int kind, long long n1, long long n2, int nn, int D, long long n,
                      long long n_edges, double *edge_list_dev, cudaStream_t s);

long long grid_row_start(int kind, long long n1, long long n2, long long row);
int launch_band_graph(const double *Xw_dev, int kind, long long n1, long long n2, int nn, int D, long long win_start,
                      long long own_start, long long own_end, long long n_window, double beta1, long long ld,
                      int32_t *nbr_id, double *nbr_w, long long *ids_dev, double *w_dev, long long *n_edges,
                      unsigned long long *wmax_bits, cudaStream_t s);

// forward-edge weights of the window nodes [0, n_fw) (implicit-grid form of phase B)
int launch_band_fwd(const double *Xw_dev, int kind, long long n1, long long n2, int nn, int D, long long win_start,
                    long long n_fw, double beta1, long long ldw, double2 *fwd, cudaStream_t s);
int launch_fwd_factor(double2 *fwd, long long count, double beta, int weighted, cudaStream_t s);

// ---- alpha-beta swap on the device (kernels_cut.cu) ---------------------------------------
// The graph in CSR form (both directions of every edge; per slot its edge number and the slot of the
// reverse arc) and the max-flow arrays of one move, for n sites, E edges and K labels.  About
// 52 bytes per site and 36 per slot (2E slots).
struct SwapScratch {
    int64_t n = 0, E = 0, bytes = 0;
    int K = 0;
    DevBuf<long long> start;                  // [n+1]
    DevBuf<long long> nbr, eid, rev, rcap;    // [2E]
    DevBuf<int32_t> wslot;                    // [2E] integer edge weight per slot
    DevBuf<long long> act, var;               // active sites; site -> compact index or -1
    DevBuf<long long> excess, inflow, tcap;   // per compact index
    DevBuf<int> h;                            // heights
    DevBuf<int32_t> V;                        // [K*K]
    DevBuf<long long> ctl;                    // control words
    MappedBuf map;                            // their host-mapped copy
};
int swap_scratch_alloc(SwapScratch &s, int64_t n, int64_t E, int K);
// the graph from a device edge list [E,2] (0 <= id1 < id2 < n)
int swap_graph_from_edges(SwapScratch &s, const long long *edge_ids, cudaStream_t st);
// the graph from a region's neighbour slots [W][ld] (-1 = empty), filled from an edge list sorted by (id1, id2)
int swap_graph_from_ell(SwapScratch &s, const int32_t *nbr_id, int W, int64_t ld, cudaStream_t st);
// GeneralGraphCut::swap(n_iter) of csrc/gco.cpp on device arrays: unary [n][K], w_edge [E], labels [n] (in: the
// start, out: the result); V_host [K*K].  PHMRF_E_UNSUPPORTED for negative weights or a non-submodular V.
int swap_run(SwapScratch &s, const int32_t *unary, const int32_t *w_edge, const int32_t *V_host, int32_t *labels,
             int n_iter, long long *energy_out, long long *energy_before_out, cudaStream_t st);

}  // namespace phmrf
