// Host side of libphmrf.so: handles, model preparation (K tiny Cholesky factorisations,
// kept on the host as the north star specifies), region upload / graph layout, and the
// extern "C" entry points declared in include/phmrf.h.
#include <atomic>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace phmrf {

static thread_local std::string g_error;
static std::atomic<long long> g_launches{0};
// One bulk transfer per direction and device at a time.  Regions driven from different threads
// (the EM driver's pool, bench.py's end-to-end leg) would otherwise share the link in each
// direction and advance in lock step -- every upload phase together, then every download phase
// together -- and never use PCIe in both directions at once.  Taking turns pipelines them: one
// region's integer cost arrays go down while the next one's features go up and its kernels run.
static std::mutex g_h2d_turn[64], g_d2h_turn[64];

void set_error(const std::string &msg) { g_error = msg; }
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    g_error = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what + " (" + file + ":" +
              std::to_string(line) + ")";
    cudaGetLastError();  // clear the sticky-less error state
    return PHMRF_E_CUDA;
}

}  // namespace phmrf

using namespace phmrf;

struct phmrf_ctx {
    int device = 0, K = 0, D = 0, sm_count = 0;
    bool has_model = false;
    bool potts = false;
    double beta = 0.0, vmax = 0.0;
    // pygco's float -> int scale factors (phmrf_set_quantiser): unary, edge weights, V
    double uprec = 100000.0, wprec = 1000.0, sprec = 100.0;
    unsigned long long version = 0;
    std::vector<double> packed;  // K * model_stride(D)
    std::vector<double> V;       // K*K
    DevBuf<double> d_model;      // K * model_stride(D) packed factors
    DevBuf<double> d_V;
};

// The stream a region runs on.  A base of phmrf_region, so that an owned stream is destroyed after the buffers.
struct RegionStream {
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    ~RegionStream() {
        if (own_stream) cudaStreamDestroy(stream);
        cudaGetLastError();  // teardown has no caller to report to
    }
};

struct phmrf_region : RegionStream {
    phmrf_ctx *ctx;
    int64_t n = 0, n_window = 0, own_offset = 0, ld = 0, E = 0;
    int W = 0;
    double wmax = 0.0;
    DevBuf<double> d_X;          // [D][ld]
    DevBuf<double> d_logp;       // tiled [ld/32][KP][32] (common.cuh lp_index)
    DevBuf<double> d_rowmax;     // [ld] max_k logp per node (written by the quantise kernel)
    DevBuf<int32_t> d_unary;     // [n][K]
    DevBuf<int32_t> d_labels;    // [n_window]
    DevBuf<int32_t> d_nbr_id;    // [W][ld]
    DevBuf<double> d_nbr_w;      // [W][ld]
    DevBuf<double> d_nbr_g;      // [W][ld] exp(beta*w), built on first use for (g_beta, g_weighted)
    // implicit-grid form (phmrf_region_create_grid): forward-edge {w, exp(beta*w)} per window node
    DevBuf<double2> d_fwd;       // [4][ldw]
    int64_t ldw = 0, own_start_gid = 0, grid_n2 = 0, grid_rows = 0;
    int grid_kind = -1, grid_nn = 0;
    double fwd_beta = 0.0;
    int fwd_weighted = -1;
    double g_beta = 0.0;
    int g_weighted = -1;
    DevBuf<double> d_edge_w;     // [E]
    DevBuf<int32_t> d_edge_wi;
    DevBuf<long long> d_edge_ids;          // [E,2] window-local, only for regions built by phmrf_region_create_grid
    DevBuf<unsigned long long> d_absmax;   // [1] bits, [1] boundary counter
    DevBuf<double> d_dwf;                  // [2] dwf, absmax
    DevBuf<long long> d_blist;
    long long bcap = 0;
    DevBuf<double> d_partials;
    DevBuf<double> d_stats;
    DevBuf<int> d_flags;
    DevBuf<long long> d_badlabel;  // [1] first out-of-range label index, -1 if none
    DevBuf<double> d_scratch;      // [K][ld] posteriors / AoS staging, allocated on demand
    int64_t scratch_elems = 0;
    bool have_logp = false, have_unary = false, have_labels = false, have_rowmax = false;
    bool edges_sorted = true;   // edge list sorted by (id1, id2): the device cut numbers the edges from the slots
    std::unique_ptr<SwapScratch> cut;  // device graph cut, allocated at the first phmrf_region_graph_cut
    int64_t bytes = 0;
    // small results (statistics, flags, dwf, counters) come back through a host-mapped buffer that a
    // kernel writes (launch_publish), not through the copy engines
    MappedBuf small;

    explicit phmrf_region(phmrf_ctx *c) : ctx(c) {}
    // The regions of one process live on different GPUs: free on the region's own, after its queued work.
    ~phmrf_region() {
        cudaSetDevice(ctx->device);
        if (stream) cudaStreamSynchronize(stream);
    }
};

// word offsets inside the mapped buffer
enum { kSmFlag = 0, kSmBadLabel = 1, kSmDwf = 2 /* 2 words */, kSmAbsmax = 4 /* 2 words */, kSmStats = 8 };

namespace {

int set_device(const phmrf_ctx *ctx) {
    PHMRF_CUDA(cudaSetDevice(ctx->device));
    return PHMRF_OK;
}

// Makes `device` current; PHMRF_E_CUDA when there is no such device, or it is not below `limit`.
int use_device(int device, const char *who, int limit = INT_MAX) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count || device >= limit) {
        cudaGetLastError();
        set_error(std::string(who) + ": no such CUDA device (this library has no CPU fallback)");
        return PHMRF_E_CUDA;
    }
    PHMRF_CUDA(cudaSetDevice(device));
    return PHMRF_OK;
}

// Lower Cholesky of a d x d matrix (row-major); false when a pivot is not positive.
bool cholesky_lower(const double *A, int d, double shift, std::vector<double> &L) {
    L.assign((size_t)d * d, 0.0);
    for (int j = 0; j < d; ++j) {
        double s = A[j * d + j] + shift;
        for (int k = 0; k < j; ++k) s -= L[j * d + k] * L[j * d + k];
        if (!(s > 0.0) || !std::isfinite(s)) return false;
        const double ljj = std::sqrt(s);
        L[j * d + j] = ljj;
        for (int i = j + 1; i < d; ++i) {
            double t = A[i * d + j];
            for (int k = 0; k < j; ++k) t -= L[i * d + k] * L[j * d + k];
            L[i * d + j] = t / ljj;
        }
    }
    return true;
}

int ensure_scratch(phmrf_region *r, int64_t elems) {
    if (r->scratch_elems >= elems) return PHMRF_OK;
    r->bytes -= r->scratch_elems * (int64_t)sizeof(double);
    r->scratch_elems = 0;
    int rc = r->d_scratch.alloc(elems, &r->bytes);
    if (rc == PHMRF_OK) r->scratch_elems = elems;
    return rc;
}

// A region on the caller's stream, or on a non-blocking stream of its own.  The region's buffers come after
// (region_alloc): a grid region counts its edges on this stream before they can be sized.
int region_open(phmrf_ctx *ctx, void *stream, std::unique_ptr<phmrf_region> &r) {
    r.reset(new phmrf_region(ctx));
    if (stream) {
        r->stream = (cudaStream_t)stream;
        return PHMRF_OK;
    }
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "cudaStreamCreate", __FILE__, __LINE__);
    r->stream = s;
    r->own_stream = true;
    return PHMRF_OK;
}

// Every buffer both region kinds share, counted in r->bytes; then X, rowmax and the log-likelihood (with its
// padding rows, common.cuh logp_rows) are cleared on the region's stream.
int region_alloc(phmrf_region *r, int64_t n_own, int64_t n_window, int64_t own_offset, int W, int64_t E) {
    const phmrf_ctx *ctx = r->ctx;
    const int K = ctx->K, D = ctx->D;
    r->n = n_own;
    r->n_window = n_window;
    r->own_offset = own_offset;
    r->W = W;
    r->E = E;
    r->ld = round_up(n_own > 0 ? n_own : 1, 64);
    r->bcap = 1 << 20;
    const int64_t ld = r->ld, stats_len = phmrf_stats_len(ctx);
    int64_t *b = &r->bytes;
    int rc;
    if ((rc = r->d_X.alloc((int64_t)D * ld, b)) || (rc = r->d_logp.alloc((int64_t)logp_rows(K) * ld, b)) ||
        (rc = r->d_rowmax.alloc(ld, b)) || (rc = r->d_unary.alloc(n_own * K, b)) ||
        (rc = r->d_labels.alloc(n_window, b)) || (rc = r->d_nbr_id.alloc((int64_t)W * ld, b)) ||
        (rc = r->d_nbr_w.alloc((int64_t)W * ld, b)) || (rc = r->d_edge_w.alloc(E, b)) ||
        (rc = r->d_edge_wi.alloc(E, b)) || (rc = r->d_absmax.alloc(2, b)) || (rc = r->d_dwf.alloc(2, b)) ||
        (rc = r->d_blist.alloc(r->bcap, b)) ||
        (rc = r->d_partials.alloc((int64_t)ctx->sm_count * ((int64_t)K * n_stat_features(D) + 3), b)) ||
        (rc = r->d_stats.alloc(stats_len, b)) || (rc = r->d_flags.alloc(1, b)) || (rc = r->d_badlabel.alloc(1, b)) ||
        (rc = r->small.alloc((size_t)(kSmStats + stats_len))))
        return rc;
    if (n_own == 0) return PHMRF_OK;
    if (cudaMemsetAsync(r->d_X, 0, sizeof(double) * D * ld, r->stream) != cudaSuccess ||
        cudaMemsetAsync(r->d_rowmax, 0, sizeof(double) * ld, r->stream) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "memset X", __FILE__, __LINE__);
    return launch_logp_init(r->d_logp, ld, K, r->stream);
}

// V as the graph cut takes it: numpy's (V * _SMOOTH_COST_PRECISION).astype(intc), K*K values
void smooth_costs_i32(const phmrf_ctx *ctx, int32_t *V_i32) {
    for (int i = 0; i < ctx->K * ctx->K; ++i) V_i32[i] = (int32_t)(ctx->V[i] * ctx->sprec);
}

// Uploads n labels and checks their range on the device (a host loop over 4e7 labels costs more than the
// copy): *first_bad is the index of the first label outside [0, K), or -1.
int upload_labels(phmrf_region *r, const int32_t *labels, int64_t n, long long *first_bad) {
    PHMRF_CUDA(cudaMemcpyAsync(r->d_labels, labels, sizeof(int32_t) * n, cudaMemcpyHostToDevice, r->stream));
    int rc;
    if ((rc = launch_check_labels(r->d_labels, n, r->ctx->K, r->d_badlabel, r->stream)) != PHMRF_OK) return rc;
    if ((rc = launch_publish(r->small.dev + kSmBadLabel, r->d_badlabel, 1, false, r->stream)) != PHMRF_OK) return rc;
    PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    *first_bad = (long long)r->small.host[kSmBadLabel];
    return PHMRF_OK;
}

// Enqueues the download of the [K][ld] array at the start of the scratch as [n,K] rows, staged behind it.
int enqueue_rows_download(phmrf_region *r, double *out) {
    if (r->n == 0) return PHMRF_OK;
    const int K = r->ctx->K;
    double *aos = r->d_scratch + (int64_t)K * r->ld;
    int rc = launch_soa_to_aos(r->d_scratch, aos, r->n, K, r->ld, r->stream);
    if (rc) return rc;
    PHMRF_CUDA(cudaMemcpyAsync(out, aos, sizeof(double) * r->n * K, cudaMemcpyDeviceToHost, r->stream));
    return PHMRF_OK;
}

}  // namespace

extern "C" {

int phmrf_abi_version(void) { return PHMRF_ABI_VERSION; }
const char *phmrf_last_error(void) { return g_error.c_str(); }
int64_t phmrf_launch_count(void) { return g_launches.load(); }

int phmrf_host_alloc(int64_t bytes, void **out) {
    if (!out || bytes < 0) {
        set_error("phmrf_host_alloc: invalid arguments");
        return PHMRF_E_INVALID;
    }
    *out = nullptr;
    // portable: usable from every device's streams (one process may drive several regions)
    PHMRF_CUDA(cudaHostAlloc(out, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocPortable));
    return PHMRF_OK;
}

int phmrf_host_free(void *p) {
    if (p) PHMRF_CUDA(cudaFreeHost(p));
    return PHMRF_OK;
}

int phmrf_ctx_create(int device, int n_states, int n_features, phmrf_ctx **out) {
    if (!out || n_states < 1 || n_features < kMinFeatures || n_features > kMaxFeatures) {
        set_error("phmrf_ctx_create: need n_states>=1 and 1<=n_features<=12");
        return n_features > kMaxFeatures ? PHMRF_E_UNSUPPORTED : PHMRF_E_INVALID;
    }
    // below 64: g_h2d_turn and g_d2h_turn hold one transfer turn per device
    int rc = use_device(device, "phmrf_ctx_create", 64);
    if (rc) return rc;
    std::unique_ptr<phmrf_ctx> ctx(new phmrf_ctx());
    ctx->device = device;
    ctx->K = n_states;
    ctx->D = n_features;
    if (cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "cudaDeviceGetAttribute", __FILE__, __LINE__);
    if ((rc = ctx->d_model.alloc((int64_t)n_states * model_stride(n_features))) ||
        (rc = ctx->d_V.alloc((int64_t)n_states * n_states)))
        return rc;
    *out = ctx.release();
    return PHMRF_OK;
}

int phmrf_ctx_destroy(phmrf_ctx *ctx) {
    if (!ctx) return PHMRF_OK;
    cudaSetDevice(ctx->device);
    delete ctx;
    return PHMRF_OK;
}

int phmrf_set_model(phmrf_ctx *ctx, const double *means, const double *covars, const double *V) {
    if (!ctx || !means || !covars || !V) {
        set_error("phmrf_set_model: null argument");
        return PHMRF_E_INVALID;
    }
    int rc = set_device(ctx);
    if (rc) return rc;
    const int K = ctx->K, D = ctx->D, PS = model_stride(D);
    std::vector<double> packed((size_t)K * PS);
    std::vector<double> L, Wm((size_t)D * D);
    const double half_log_2pi_d = 0.5 * D * std::log(2.0 * M_PI);
    const double rs2 = std::sqrt(0.5);
    for (int k = 0; k < K; ++k) {
        const double *cv = covars + (size_t)k * D * D;
        for (int i = 0; i < D; ++i)
            for (int j = 0; j < i; ++j)
                if (!(std::fabs(cv[i * D + j] - cv[j * D + i]) <= 1e-8 + 1e-5 * std::fabs(cv[j * D + i]))) {
                    set_error("'covars' must be symmetric, positive-definite");
                    return PHMRF_E_NOT_SPD;
                }
        // sklearn 0.18: cholesky(cv), on failure cholesky(cv + 1e-7*I), on failure ValueError
        if (!cholesky_lower(cv, D, 0.0, L) && !cholesky_lower(cv, D, 1e-7, L)) {
            set_error("'covars' must be symmetric, positive-definite");
            return PHMRF_E_NOT_SPD;
        }
        double logdet = 0.0;
        for (int i = 0; i < D; ++i) logdet += std::log(L[i * D + i]);
        logdet *= 2.0;
        // W = L^-1 by forward substitution, column by column
        std::fill(Wm.begin(), Wm.end(), 0.0);
        for (int c = 0; c < D; ++c) {
            for (int i = c; i < D; ++i) {
                double s = (i == c) ? 1.0 : 0.0;
                for (int j = c; j < i; ++j) s -= L[i * D + j] * Wm[j * D + c];
                Wm[i * D + c] = s / L[i * D + i];
            }
        }
        double *p = packed.data() + (size_t)k * PS;
        const double *mu = means + (size_t)k * D;
        p[0] = half_log_2pi_d + 0.5 * logdet;
        int q = 1;
        for (int i = 0; i < D; ++i) {
            double ci = 0.0;
            for (int j = 0; j <= i; ++j) ci += rs2 * Wm[i * D + j] * mu[j];
            p[q++] = ci;
            for (int j = 0; j <= i; ++j) p[q++] = rs2 * Wm[i * D + j];
        }
    }
    // label compatibility: Potts beta*(1-I) (phylo_hmrf.py:524-536) takes the fast path
    bool potts = true;
    double beta = K > 1 ? V[1] : 0.0, vmax = V[0];
    for (int i = 0; i < K; ++i)
        for (int j = 0; j < K; ++j) {
            const double v = V[i * K + j];
            if (v > vmax || std::isnan(v)) vmax = v;
            if (i == j ? v != 0.0 : v != beta) potts = false;
        }
    if (!(beta >= 0.0)) potts = false;
    ctx->packed.swap(packed);
    ctx->V.assign(V, V + (size_t)K * K);
    ctx->potts = potts;
    ctx->beta = beta;
    ctx->vmax = vmax;
    ctx->version++;
    ctx->has_model = true;
    PHMRF_CUDA(cudaDeviceSynchronize());
    PHMRF_CUDA(cudaMemcpy(ctx->d_model, ctx->packed.data(), sizeof(double) * ctx->packed.size(),
                          cudaMemcpyHostToDevice));
    PHMRF_CUDA(cudaMemcpy(ctx->d_V, ctx->V.data(), sizeof(double) * ctx->V.size(), cudaMemcpyHostToDevice));
    return PHMRF_OK;
}

int phmrf_set_quantiser(phmrf_ctx *ctx, double unary_precision, double pairwise_precision, double smooth_precision) {
    // |scaled value| must stay below 2^31 for the int32 conversion; pygco's own limit is GCO's 1e7 per term
    if (!ctx || !(unary_precision >= 1.0 && unary_precision <= 1e9) ||
        !(pairwise_precision >= 1.0 && pairwise_precision <= 1e9) ||
        !(smooth_precision >= 1.0 && smooth_precision <= 1e9)) {
        set_error("phmrf_set_quantiser: precisions must lie in [1, 1e9]");
        return PHMRF_E_INVALID;
    }
    ctx->uprec = unary_precision;
    ctx->wprec = pairwise_precision;
    ctx->sprec = smooth_precision;
    return PHMRF_OK;
}

int phmrf_get_quantiser(const phmrf_ctx *ctx, double *unary_precision, double *pairwise_precision,
                        double *smooth_precision) {
    if (!ctx) return PHMRF_E_INVALID;
    if (unary_precision) *unary_precision = ctx->uprec;
    if (pairwise_precision) *pairwise_precision = ctx->wprec;
    if (smooth_precision) *smooth_precision = ctx->sprec;
    return PHMRF_OK;
}

int phmrf_region_create(phmrf_ctx *ctx, const double *X, int64_t n_own, int64_t n_window, int64_t own_offset,
                        const int64_t *edge_ids, const double *edge_w, int64_t n_edges, void *stream,
                        phmrf_region **out) {
    if (!ctx || !out || n_own < 0 || n_window < n_own || own_offset < 0 || own_offset + n_own > n_window ||
        n_edges < 0 || (n_own > 0 && !X) || (n_edges > 0 && (!edge_ids || !edge_w)) ||
        n_window >= ((int64_t)1 << 31)) {
        set_error("phmrf_region_create: invalid shape arguments");
        return PHMRF_E_INVALID;
    }
    int rc = set_device(ctx);
    if (rc) return rc;
    const int D = ctx->D;
    // ---- graph layout on the host: per owned node, its neighbours in ascending edge order
    std::vector<int> deg((size_t)n_own, 0);
    double wmax = 0.0;
    bool sorted = true;
    for (int64_t e = 0; e < n_edges; ++e) {
        const int64_t a = edge_ids[2 * e], b = edge_ids[2 * e + 1];
        if (a < 0 || b < 0 || a >= n_window || b >= n_window || a == b) {
            set_error("phmrf_region_create: edge id out of range (or self loop) at edge " + std::to_string(e));
            return PHMRF_E_INVALID;
        }
        if (a > b || (e > 0 && (edge_ids[2 * e - 2] > a || (edge_ids[2 * e - 2] == a && edge_ids[2 * e - 1] > b))))
            sorted = false;
        if (a >= own_offset && a < own_offset + n_own) deg[a - own_offset]++;
        if (b >= own_offset && b < own_offset + n_own) deg[b - own_offset]++;
        const double aw = std::fabs(edge_w[e]);
        if (aw > wmax || std::isnan(aw)) wmax = aw;
    }
    int W = 0;
    for (int64_t i = 0; i < n_own; ++i) W = deg[i] > W ? deg[i] : W;

    std::unique_ptr<phmrf_region> r;
    if ((rc = region_open(ctx, stream, r)) || (rc = region_alloc(r.get(), n_own, n_window, own_offset, W, n_edges)))
        return rc;
    r->wmax = wmax;
    r->edges_sorted = sorted;
    const int64_t ld = r->ld;
    // X: upload row-major, transpose on the device into the feature-major layout
    if (n_own > 0) {
        if ((rc = ensure_scratch(r.get(), n_own * D)) != PHMRF_OK) return rc;
        if (cudaMemcpyAsync(r->d_scratch, X, sizeof(double) * n_own * D, cudaMemcpyHostToDevice, r->stream) !=
            cudaSuccess)
            return cuda_fail(cudaGetLastError(), "upload X", __FILE__, __LINE__);
        if ((rc = launch_aos_to_soa(r->d_scratch, r->d_X, n_own, D, ld, r->stream)) != PHMRF_OK) return rc;
    }
    if (W > 0) {
        std::vector<int32_t> nid((size_t)W * ld, -1);
        std::vector<double> nw((size_t)W * ld, 0.0);
        std::vector<int> fill((size_t)n_own, 0);
        for (int64_t e = 0; e < n_edges; ++e) {
            const int64_t a = edge_ids[2 * e], b = edge_ids[2 * e + 1];
            if (a >= own_offset && a < own_offset + n_own) {
                const int64_t i = a - own_offset;
                const int s = fill[i]++;
                nid[(size_t)s * ld + i] = (int32_t)b;
                nw[(size_t)s * ld + i] = edge_w[e];
            }
            if (b >= own_offset && b < own_offset + n_own) {
                const int64_t i = b - own_offset;
                const int s = fill[i]++;
                nid[(size_t)s * ld + i] = (int32_t)a;
                nw[(size_t)s * ld + i] = edge_w[e];
            }
        }
        if (cudaMemcpy(r->d_nbr_id, nid.data(), sizeof(int32_t) * nid.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(r->d_nbr_w, nw.data(), sizeof(double) * nw.size(), cudaMemcpyHostToDevice) != cudaSuccess)
            return cuda_fail(cudaGetLastError(), "upload graph", __FILE__, __LINE__);
    }
    if (n_edges > 0 &&
        cudaMemcpy(r->d_edge_w, edge_w, sizeof(double) * n_edges, cudaMemcpyHostToDevice) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "upload edge weights", __FILE__, __LINE__);
    if (cudaStreamSynchronize(r->stream) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "region upload", __FILE__, __LINE__);
    *out = r.release();
    return PHMRF_OK;
}

int phmrf_region_create_grid(phmrf_ctx *ctx, const double *X_window, int kind, int64_t n1, int64_t n2, int64_t row0,
                             int64_t row1, int num_neighbor, double beta1, void *stream, phmrf_region **out) {
    const int64_t rows = kind == 1 ? n2 : n1;
    if (!ctx || !out || !X_window || (kind != 0 && kind != 1) || n1 < 1 || n2 < 1 || (kind == 1 && n1 != n2) ||
        (num_neighbor != 8 && num_neighbor != 4) || row0 < 0 || row1 <= row0 || row1 > rows) {
        set_error("phmrf_region_create_grid: invalid geometry (kind 0/1, num_neighbor 8/4, 0 <= row0 < row1 <= rows)");
        return PHMRF_E_INVALID;
    }
    int rc = set_device(ctx);
    if (rc) return rc;
    const int D = ctx->D;
    const int64_t h0 = row0 > 0 ? row0 - 1 : 0, h1 = row1 < rows ? row1 + 1 : rows;
    const int64_t win_start = grid_row_start(kind, n1, n2, h0), win_end = grid_row_start(kind, n1, n2, h1);
    const int64_t own_start = grid_row_start(kind, n1, n2, row0), own_end = grid_row_start(kind, n1, n2, row1);
    const int64_t n_window = win_end - win_start, n_own = own_end - own_start;
    if (n_window >= ((int64_t)1 << 31)) {
        set_error("phmrf_region_create_grid: window too large for 32-bit neighbour ids");
        return PHMRF_E_INVALID;
    }
    std::unique_ptr<phmrf_region> r;
    if ((rc = region_open(ctx, stream, r)) != PHMRF_OK) return rc;
    DevBuf<double> dXw;  // the window's features [n_window, D], only while the region is built
    if ((rc = dXw.alloc(n_window * D)) != PHMRF_OK) return rc;
    if (cudaMemcpyAsync(dXw, X_window, sizeof(double) * n_window * D, cudaMemcpyHostToDevice, r->stream) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "upload X window", __FILE__, __LINE__);
    long long n_edges = 0;  // the counting call: the edge count sizes the edge buffers
    if ((rc = launch_band_graph(dXw, kind, n1, n2, num_neighbor, D, win_start, own_start, own_end, n_window, beta1, 0,
                                nullptr, nullptr, nullptr, nullptr, &n_edges, nullptr, r->stream)) ||
        (rc = region_alloc(r.get(), n_own, n_window, own_start - win_start, num_neighbor, n_edges)) ||
        (rc = r->d_edge_ids.alloc(2 * n_edges, &r->bytes)))
        return rc;
    if ((rc = launch_aos_to_soa(dXw + r->own_offset * D, r->d_X, n_own, D, r->ld, r->stream)) != PHMRF_OK) return rc;
    // implicit-grid form of phase B: one {w, g} pair per forward edge of every window node up to the last owned one
    r->grid_kind = kind;
    r->grid_nn = num_neighbor;
    r->grid_n2 = n2;
    r->grid_rows = rows;
    r->own_start_gid = own_start;
    r->ldw = round_up(r->own_offset + n_own > 0 ? r->own_offset + n_own : 1, 64);
    if ((rc = r->d_fwd.alloc(4 * r->ldw, &r->bytes)) != PHMRF_OK) return rc;
    if (cudaMemsetAsync(r->d_fwd, 0, sizeof(double2) * 4 * r->ldw, r->stream) != cudaSuccess)  // incl. the row padding
        return cuda_fail(cudaGetLastError(), "memset forward weights", __FILE__, __LINE__);
    if ((rc = launch_band_fwd(dXw, kind, n1, n2, num_neighbor, D, win_start, r->own_offset + n_own, beta1, r->ldw,
                              r->d_fwd, r->stream)) != PHMRF_OK)
        return rc;
    // max|w| lands in d_absmax[1] (free until the first quantise resets it as the boundary counter)
    if ((rc = launch_band_graph(dXw, kind, n1, n2, num_neighbor, D, win_start, own_start, own_end, n_window, beta1,
                                r->ld, r->d_nbr_id, r->d_nbr_w, r->d_edge_ids, r->d_edge_w, &n_edges, r->d_absmax + 1,
                                r->stream)) != PHMRF_OK)
        return rc;
    unsigned long long wbits = 0;
    if (cudaMemcpy(&wbits, r->d_absmax + 1, sizeof(wbits), cudaMemcpyDeviceToHost) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "read max|w|", __FILE__, __LINE__);
    std::memcpy(&r->wmax, &wbits, sizeof(double));
    *out = r.release();
    return PHMRF_OK;
}

int64_t phmrf_region_n_edges(const phmrf_region *r) { return r ? r->E : 0; }
int64_t phmrf_region_n_own(const phmrf_region *r) { return r ? r->n : 0; }
int64_t phmrf_region_n_window(const phmrf_region *r) { return r ? r->n_window : 0; }
int64_t phmrf_region_own_offset(const phmrf_region *r) { return r ? r->own_offset : 0; }

int phmrf_region_edges(phmrf_region *r, int64_t *edge_ids_out, double *edge_w_out) {
    if (!r) return PHMRF_E_INVALID;
    if (!r->d_edge_ids) {
        set_error("phmrf_region_edges: only regions built by phmrf_region_create_grid keep their edge list");
        return PHMRF_E_STATE;
    }
    int rc = set_device(r->ctx);
    if (rc) return rc;
    if (r->E > 0) {
        if (edge_ids_out)
            PHMRF_CUDA(cudaMemcpy(edge_ids_out, r->d_edge_ids, sizeof(long long) * 2 * r->E, cudaMemcpyDeviceToHost));
        if (edge_w_out) PHMRF_CUDA(cudaMemcpy(edge_w_out, r->d_edge_w, sizeof(double) * r->E, cudaMemcpyDeviceToHost));
    }
    return PHMRF_OK;
}

int phmrf_region_set_edge_weights(phmrf_region *r, const double *edge_w, int64_t n_edges) {
    if (!r || (n_edges > 0 && !edge_w) || n_edges != r->E) {
        set_error("phmrf_region_set_edge_weights: need the region's own number of edge weights");
        return PHMRF_E_INVALID;
    }
    if (!r->d_fwd) {
        set_error("phmrf_region_set_edge_weights: only for regions built by phmrf_region_create_grid");
        return PHMRF_E_STATE;
    }
    int rc = set_device(r->ctx);
    if (rc) return rc;
    double wmax = 0.0;
    for (int64_t e = 0; e < n_edges; ++e) {
        const double aw = std::fabs(edge_w[e]);
        if (aw > wmax || std::isnan(aw)) wmax = aw;
    }
    if (n_edges > 0) {
        PHMRF_CUDA(cudaMemcpyAsync(r->d_edge_w, edge_w, sizeof(double) * n_edges, cudaMemcpyHostToDevice, r->stream));
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    }
    r->wmax = wmax;
    r->have_unary = false;
    return PHMRF_OK;
}

int phmrf_region_update_X(phmrf_region *r, const double *X) {
    if (!r || (!X && r->n > 0)) return PHMRF_E_INVALID;
    int rc = set_device(r->ctx);
    if (rc) return rc;
    if (r->n == 0) return PHMRF_OK;
    const int D = r->ctx->D;
    if ((rc = ensure_scratch(r, r->n * D)) != PHMRF_OK) return rc;
    {
        std::lock_guard<std::mutex> turn(g_h2d_turn[r->ctx->device]);
        PHMRF_CUDA(cudaMemcpyAsync(r->d_scratch, X, sizeof(double) * r->n * D, cudaMemcpyHostToDevice, r->stream));
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));  // X may be reused by the caller; the turn ends with the copy
    }
    if ((rc = launch_aos_to_soa(r->d_scratch, r->d_X, r->n, D, r->ld, r->stream)) != PHMRF_OK) return rc;
    r->have_logp = false;
    r->have_unary = false;
    return PHMRF_OK;
}

int phmrf_region_destroy(phmrf_region *r) {
    delete r;
    return PHMRF_OK;
}

int phmrf_region_sync(phmrf_region *r) {
    if (!r) return PHMRF_E_INVALID;
    PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    return PHMRF_OK;
}

int64_t phmrf_region_device_bytes(const phmrf_region *r) { return r ? r->bytes : 0; }

int64_t phmrf_stats_len(const phmrf_ctx *ctx) {
    return ctx ? (int64_t)ctx->K * (1 + ctx->D + ctx->D * ctx->D) + 3 : 0;
}

void *phmrf_stats_device_ptr(phmrf_region *r) { return r ? (void *)r->d_stats.get() : nullptr; }
void *phmrf_absmax_device_ptr(phmrf_region *r) { return r ? (void *)r->d_absmax.get() : nullptr; }
double phmrf_region_weight_max(const phmrf_region *r) { return r ? r->wmax : 0.0; }
int phmrf_region_set_weight_max(phmrf_region *r, double wmax) {
    if (!r || !(wmax >= 0.0)) return PHMRF_E_INVALID;
    r->wmax = wmax;
    return PHMRF_OK;
}

// ---------------------------------------------------------------- phase A
int phmrf_emit_loglik_async(phmrf_region *r) {
    if (!r) return PHMRF_E_INVALID;
    phmrf_ctx *ctx = r->ctx;
    if (!ctx->has_model) {
        set_error("phmrf_emit_loglik: phmrf_set_model has not been called");
        return PHMRF_E_STATE;
    }
    int rc = set_device(ctx);
    if (rc) return rc;
    rc = launch_emit(r->d_X, r->n, r->ld, ctx->D, ctx->K, ctx->d_model, r->d_logp, r->d_absmax, ctx->sm_count,
                     r->stream);
    if (rc == PHMRF_OK) {
        r->have_logp = true;
        r->have_unary = false;
        r->have_rowmax = false;
    }
    return rc;
}

int phmrf_emit_loglik(phmrf_region *r, double *absmax_out) {
    int rc = phmrf_emit_loglik_async(r);
    if (rc) return rc;
    if (absmax_out) {
        if ((rc = launch_publish(r->small.dev + kSmAbsmax, r->d_absmax, 1, false, r->stream)) != PHMRF_OK) return rc;
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));
        std::memcpy(absmax_out, r->small.host + kSmAbsmax, sizeof(double));
    }
    return PHMRF_OK;
}

int phmrf_get_logprob(phmrf_region *r, double *logprob_out) {
    if (!r || !logprob_out) return PHMRF_E_INVALID;
    if (!r->have_logp) {
        set_error("phmrf_get_logprob: call phmrf_emit_loglik first");
        return PHMRF_E_STATE;
    }
    int rc = set_device(r->ctx);
    if (rc) return rc;
    if (r->n == 0) return PHMRF_OK;
    const int K = r->ctx->K;
    if ((rc = ensure_scratch(r, r->n * K)) != PHMRF_OK) return rc;
    if ((rc = launch_logp_to_aos(r->d_logp, r->d_scratch, r->n, K, r->stream)) != PHMRF_OK) return rc;
    PHMRF_CUDA(cudaMemcpyAsync(logprob_out, r->d_scratch, sizeof(double) * r->n * K, cudaMemcpyDeviceToHost,
                               r->stream));
    PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    return PHMRF_OK;
}

int phmrf_quantise_async(phmrf_region *r, double dwf_in, double tol) {
    if (!r) return PHMRF_E_INVALID;
    if (!r->have_logp) {
        set_error("phmrf_quantise: call phmrf_emit_loglik first");
        return PHMRF_E_STATE;
    }
    phmrf_ctx *ctx = r->ctx;
    int rc = set_device(ctx);
    if (rc) return rc;
    if ((rc = launch_dwf(r->d_absmax, r->wmax, ctx->vmax, dwf_in, r->d_dwf, r->stream)) != PHMRF_OK) return rc;
    // one launch: integer unary + per-node max + integer edge weights (pygco converts the edge
    // weights on every call, the down-weight factor changes with the model)
    if ((rc = launch_quantise(r->d_logp, r->n, ctx->K, r->d_dwf, tol, ctx->uprec, r->d_unary, r->d_rowmax, r->d_blist,
                              r->bcap, r->d_absmax + 1, r->E > 0 ? r->d_edge_w.get() : nullptr, r->E, ctx->wprec,
                              r->d_edge_wi, ctx->sm_count, r->stream)) != PHMRF_OK)
        return rc;
    r->have_unary = true;
    r->have_rowmax = true;
    return PHMRF_OK;
}

int phmrf_quantise(phmrf_region *r, double dwf_in, double tol, int32_t *unary_i32_out, int32_t *w_i32_out,
                   int32_t *V_i32_out, double *dwf_out, int64_t *boundary_idx, int64_t boundary_cap,
                   int64_t *n_boundary) {
    int rc = phmrf_quantise_async(r, dwf_in, tol);
    if (rc) return rc;
    phmrf_ctx *ctx = r->ctx;
    const int K = ctx->K;
    double dwf2[2] = {0, 0};
    unsigned long long nb = 0;
    if ((w_i32_out && r->E > 0) || (unary_i32_out && r->n > 0)) {
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));  // the kernels first: a turn is spent on copying only
        std::lock_guard<std::mutex> turn(g_d2h_turn[ctx->device]);
        if (w_i32_out && r->E > 0)
            PHMRF_CUDA(cudaMemcpyAsync(w_i32_out, r->d_edge_wi, sizeof(int32_t) * r->E, cudaMemcpyDeviceToHost, r->stream));
        if (unary_i32_out && r->n > 0)
            PHMRF_CUDA(cudaMemcpyAsync(unary_i32_out, r->d_unary, sizeof(int32_t) * r->n * K, cudaMemcpyDeviceToHost,
                                       r->stream));
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    }
    if ((rc = launch_publish(r->small.dev + kSmDwf, r->d_dwf, 2, false, r->stream)) != PHMRF_OK) return rc;
    if ((rc = launch_publish(r->small.dev + kSmAbsmax, r->d_absmax, 2, false, r->stream)) != PHMRF_OK) return rc;
    PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    std::memcpy(dwf2, r->small.host + kSmDwf, sizeof(dwf2));
    nb = r->small.host[kSmAbsmax + 1];
    if (dwf_out) *dwf_out = dwf2[0];
    if (n_boundary) *n_boundary = (int64_t)nb;
    if (boundary_idx && boundary_cap > 0 && nb > 0) {
        int64_t m = (int64_t)nb < boundary_cap ? (int64_t)nb : boundary_cap;
        if (m > r->bcap) m = r->bcap;
        PHMRF_CUDA(cudaMemcpy(boundary_idx, r->d_blist, sizeof(long long) * m, cudaMemcpyDeviceToHost));
    }
    if (V_i32_out) smooth_costs_i32(ctx, V_i32_out);
    return PHMRF_OK;
}

// ---------------------------------------------------------------- phase B
int phmrf_set_labels(phmrf_region *r, const int32_t *labels_window) {
    if (!r || !labels_window) return PHMRF_E_INVALID;
    int rc = set_device(r->ctx);
    if (rc) return rc;
    long long first_bad = -1;
    if ((rc = upload_labels(r, labels_window, r->n_window, &first_bad)) != PHMRF_OK) return rc;
    if (first_bad >= 0) {
        r->have_labels = false;
        set_error("phmrf_set_labels: label out of range at node " + std::to_string(first_bad));
        return PHMRF_E_INVALID;
    }
    r->have_labels = true;
    return PHMRF_OK;
}

int phmrf_labels_argmin_unary(phmrf_region *r, int32_t *labels_out) {
    if (!r) return PHMRF_E_INVALID;
    if (!r->have_unary || r->n != r->n_window) {
        set_error("phmrf_labels_argmin_unary: needs the integer unary of a whole region");
        return PHMRF_E_STATE;
    }
    int rc = set_device(r->ctx);
    if (rc) return rc;
    if ((rc = launch_argmin_unary(r->d_unary, r->n, r->ctx->K, r->d_labels, r->stream)) != PHMRF_OK) return rc;
    r->have_labels = true;
    if (labels_out && r->n > 0) {
        PHMRF_CUDA(cudaMemcpyAsync(labels_out, r->d_labels, sizeof(int32_t) * r->n, cudaMemcpyDeviceToHost, r->stream));
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    }
    return PHMRF_OK;
}

// overflow_redo: the redo after the pipeline kernel flagged a soft-max overflow, always on the general kernel
static int estep_enqueue(phmrf_region *r, int estimate_type, bool want_post, bool want_pp = false,
                         bool overflow_redo = false) {
    if (!r) return PHMRF_E_INVALID;
    if (!r->have_logp || !r->have_labels) {
        set_error("phmrf_estep_stats: needs phmrf_emit_loglik and labels first");
        return PHMRF_E_STATE;
    }
    phmrf_ctx *ctx = r->ctx;
    int rc = set_device(ctx);
    if (rc) return rc;
    EstepArgs a;
    a.X_soa = r->d_X;
    a.logp = r->d_logp;
    a.rowmax = r->d_rowmax;
    if (!r->have_rowmax) {  // a log-likelihood the quantise kernel has not seen
        if ((rc = launch_rowmax(r->d_logp, r->n, ctx->K, r->d_rowmax, nullptr, r->stream)) != PHMRF_OK) return rc;
        r->have_rowmax = true;
    }
    a.labels = r->d_labels;
    a.nbr_id = r->d_nbr_id;
    a.nbr_w = r->d_nbr_w;
    a.V = ctx->d_V;
    a.beta = ctx->beta;
    a.potts = ctx->potts ? 1 : 0;
    a.n = r->n;
    a.ld = r->ld;
    a.own_offset = r->own_offset;
    a.D = ctx->D;
    a.K = ctx->K;
    a.W = r->W;
    a.estimate_type = estimate_type;
    a.post_soa = nullptr;
    a.pp_soa = nullptr;
    if (want_post || want_pp) {
        if ((rc = ensure_scratch(r, (int64_t)ctx->K * r->ld + r->n * ctx->K)) != PHMRF_OK) return rc;
        if (want_post) a.post_soa = r->d_scratch;
        if (want_pp) a.pp_soa = r->d_scratch;
    }
    a.partials = r->d_partials;
    a.stats_out = r->d_stats;
    a.flags = r->d_flags;
    a.s_bound = ctx->beta * r->W * (estimate_type == 3 ? r->wmax : 1.0);
    a.nbr_g = nullptr;
    a.exp_beta = std::exp(ctx->beta);
    a.fwd_wg = nullptr;
    a.ldw = r->ldw;
    a.grid_kind = -1;
    a.grid_nn = r->grid_nn;
    a.grid_n2 = r->grid_n2;
    a.grid_rows = r->grid_rows;
    a.own_start_gid = r->own_start_gid;
    const bool bulk = !overflow_redo && estep_bulk_supported(a);
    if (bulk) {
        // per-slot factors of the pipeline kernel: constant while beta and the weights are
        const int weighted = estimate_type == 3 ? 1 : 0;
        if (r->d_fwd) {
            // region built from the grid geometry: implicit neighbours, each weight stored once
            if (r->fwd_weighted != weighted || r->fwd_beta != ctx->beta) {
                if ((rc = launch_fwd_factor(r->d_fwd, 4 * r->ldw, ctx->beta, weighted, r->stream)) != PHMRF_OK) return rc;
                r->fwd_weighted = weighted;
                r->fwd_beta = ctx->beta;
            }
            a.fwd_wg = r->d_fwd;
            a.grid_kind = r->grid_kind;
        } else {
            if (!r->d_nbr_g) {
                if ((rc = r->d_nbr_g.alloc((int64_t)r->W * r->ld, &r->bytes)) != PHMRF_OK) return rc;
                r->g_weighted = -1;
            }
            if (r->g_weighted != weighted || r->g_beta != ctx->beta) {
                if ((rc = launch_nbr_g(r->d_nbr_id, r->d_nbr_w, r->d_nbr_g, (int64_t)r->W * r->ld, ctx->beta, weighted,
                                       r->stream)) != PHMRF_OK)
                    return rc;
                r->g_weighted = weighted;
                r->g_beta = ctx->beta;
            }
            a.nbr_g = r->d_nbr_g;
        }
    }
    PHMRF_CUDA(cudaMemsetAsync(r->d_flags, 0, sizeof(int), r->stream));
    return bulk ? launch_estep_bulk(a, ctx->sm_count, r->stream) : launch_estep(a, ctx->sm_count, r->stream);
}

int phmrf_estep_stats_async(phmrf_region *r, int estimate_type) { return estep_enqueue(r, estimate_type, false); }

int phmrf_estep_stats(phmrf_region *r, int estimate_type, double *post_out, double *stats_out,
                      double *cost_sums_out) {
    int rc = estep_enqueue(r, estimate_type, post_out != nullptr);
    if (rc) return rc;
    const int64_t len = phmrf_stats_len(r->ctx);
    std::vector<double> host((size_t)len);
    for (int attempt = 0; attempt < 2; ++attempt) {
        int flag = 0;
        if (post_out && (rc = enqueue_rows_download(r, post_out)) != PHMRF_OK) return rc;
        if ((rc = launch_publish(r->small.dev + kSmStats, r->d_stats, (int)len, false, r->stream)) != PHMRF_OK) return rc;
        if ((rc = launch_publish(r->small.dev + kSmFlag, r->d_flags, 1, true, r->stream)) != PHMRF_OK) return rc;
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));
        std::memcpy(host.data(), r->small.host + kSmStats, sizeof(double) * len);
        flag = (int)(long long)r->small.host[kSmFlag];
        if (!(flag & 1) || attempt == 1) break;
        // the pipeline kernel met a soft-max overflow (only reachable with extreme beta):
        // redo the region on the general kernel, which uses the exact maximum
        if ((rc = estep_enqueue(r, estimate_type, post_out != nullptr, false, true)) != PHMRF_OK) return rc;
    }
    if (stats_out) std::memcpy(stats_out, host.data(), sizeof(double) * (len - 3));
    if (cost_sums_out) std::memcpy(cost_sums_out, host.data() + (len - 3), sizeof(double) * 3);
    return PHMRF_OK;
}

int phmrf_pairwise_potential(phmrf_region *r, int estimate_type, double *pp_out) {
    if (!r || !pp_out) return PHMRF_E_INVALID;
    int rc = estep_enqueue(r, estimate_type, false, true);
    if (rc || (rc = enqueue_rows_download(r, pp_out))) return rc;
    PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    return PHMRF_OK;
}

int phmrf_set_logprob(phmrf_region *r, const double *logprob) {
    if (!r || !logprob) return PHMRF_E_INVALID;
    int rc = set_device(r->ctx);
    if (rc) return rc;
    const int K = r->ctx->K;
    if (r->n > 0) {
        if ((rc = ensure_scratch(r, r->n * K)) != PHMRF_OK) return rc;
        PHMRF_CUDA(cudaMemcpyAsync(r->d_scratch, logprob, sizeof(double) * r->n * K, cudaMemcpyHostToDevice, r->stream));
        if ((rc = launch_logp_from_aos(r->d_scratch, r->d_logp, r->n, K, r->stream)) != PHMRF_OK) return rc;
    }
    // max|logp| (the data term of the down-weight factor) and the per-node maxima follow the new array
    PHMRF_CUDA(cudaMemsetAsync(r->d_absmax, 0, sizeof(unsigned long long), r->stream));
    if ((rc = launch_rowmax(r->d_logp, r->n, K, r->d_rowmax, r->d_absmax, r->stream)) != PHMRF_OK) return rc;
    PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    r->have_logp = true;
    r->have_unary = false;
    r->have_rowmax = true;
    return PHMRF_OK;
}

// ---------------------------------------------------------------- graph cut on the device
int phmrf_graph_cut_swap(int device, int64_t n_sites, int32_t n_labels, const int32_t *unary, const int64_t *edge_ids,
                         const int32_t *edge_w, int64_t n_edges, const int32_t *smooth, const int32_t *init_labels,
                         int32_t n_iter, int32_t *labels_out, long long *energy_out, long long *energy_before_out) {
    if (n_sites <= 0 || n_labels <= 0 || !unary || !smooth || !labels_out || n_edges < 0 ||
        (n_edges > 0 && (!edge_ids || !edge_w))) {
        set_error("GCO (device swap) phmrf_graph_cut_swap: invalid arguments");
        return PHMRF_E_INVALID;
    }
    for (int64_t e = 0; e < n_edges; ++e) {
        const int64_t a = edge_ids[2 * e], b = edge_ids[2 * e + 1];
        if (a < 0 || b < 0 || a >= n_sites || b >= n_sites || a >= b) {
            set_error("GCO (device swap) phmrf_graph_cut_swap: edges must satisfy 0 <= id1 < id2 < n_sites");
            return PHMRF_E_INVALID;
        }
    }
    if (init_labels)
        for (int64_t i = 0; i < n_sites; ++i)
            if (init_labels[i] < 0 || init_labels[i] >= n_labels) {
                set_error("GCO (device swap) phmrf_graph_cut_swap: init label out of range");
                return PHMRF_E_INVALID;
            }
    int rc = use_device(device, "GCO (device swap) phmrf_graph_cut_swap");
    if (rc) return rc;
    SwapScratch s;
    DevBuf<int32_t> d_unary, d_labels, d_w;
    DevBuf<long long> d_ids;
    if ((rc = swap_scratch_alloc(s, n_sites, n_edges, n_labels)) || (rc = d_unary.alloc(n_sites * n_labels)) ||
        (rc = d_labels.alloc(n_sites)) || (rc = d_w.alloc(n_edges)) || (rc = d_ids.alloc(2 * n_edges)))
        return rc;
    cudaStream_t st = nullptr;
    PHMRF_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    const size_t nu = sizeof(int32_t) * (size_t)n_sites * n_labels;
    if (cudaMemcpyAsync(d_unary, unary, nu, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        (n_edges > 0 &&
         (cudaMemcpyAsync(d_w, edge_w, sizeof(int32_t) * n_edges, cudaMemcpyHostToDevice, st) != cudaSuccess ||
          cudaMemcpyAsync(d_ids, edge_ids, sizeof(long long) * 2 * n_edges, cudaMemcpyHostToDevice, st) !=
              cudaSuccess)) ||
        (init_labels ? cudaMemcpyAsync(d_labels, init_labels, sizeof(int32_t) * n_sites, cudaMemcpyHostToDevice, st)
                     : cudaMemsetAsync(d_labels, 0, sizeof(int32_t) * n_sites, st)) != cudaSuccess)
        rc = cuda_fail(cudaGetLastError(), "graph cut upload", __FILE__, __LINE__);
    if (rc == PHMRF_OK) rc = swap_graph_from_edges(s, d_ids, st);
    if (rc == PHMRF_OK) rc = swap_run(s, d_unary, d_w, smooth, d_labels, n_iter, energy_out, energy_before_out, st);
    if (rc == PHMRF_OK &&
        (cudaMemcpyAsync(labels_out, d_labels, sizeof(int32_t) * n_sites, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
         cudaStreamSynchronize(st) != cudaSuccess))
        rc = cuda_fail(cudaGetLastError(), "graph cut download", __FILE__, __LINE__);
    cudaStreamSynchronize(st);  // before the buffers go
    cudaStreamDestroy(st);
    return rc;
}

int phmrf_region_graph_cut(phmrf_region *r, const int32_t *init_labels, int32_t n_iter, int32_t *labels_out,
                           long long *energy_out, long long *energy_before_out) {
    if (!r) return PHMRF_E_INVALID;
    if (r->n != r->n_window || r->n == 0) {
        set_error("GCO (device swap) phmrf_region_graph_cut: needs a whole, non-empty region (a band's cut needs the other bands' unary)");
        return PHMRF_E_INVALID;
    }
    if (!r->edges_sorted) {
        set_error("GCO (device swap) phmrf_region_graph_cut: the region's edge list is not sorted by (id1, id2)");
        return PHMRF_E_INVALID;
    }
    if (!r->have_unary) {
        set_error("GCO (device swap) phmrf_region_graph_cut: call phmrf_quantise first");
        return PHMRF_E_STATE;
    }
    phmrf_ctx *ctx = r->ctx;
    int rc = set_device(ctx);
    if (rc) return rc;
    const int K = ctx->K;
    if (!r->cut) {
        std::unique_ptr<SwapScratch> cut(new SwapScratch());
        if ((rc = swap_scratch_alloc(*cut, r->n, r->E, K)) ||
            (rc = swap_graph_from_ell(*cut, r->d_nbr_id, r->W, r->ld, r->stream)))
            return rc;
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));
        r->bytes += cut->bytes;
        r->cut = std::move(cut);
    }
    r->have_labels = false;
    if (init_labels) {
        long long first_bad = -1;
        if ((rc = upload_labels(r, init_labels, r->n, &first_bad)) != PHMRF_OK) return rc;
        if (first_bad >= 0) {
            set_error("GCO (device swap) phmrf_region_graph_cut: init label out of range at node " + std::to_string(first_bad));
            return PHMRF_E_INVALID;
        }
    } else {
        PHMRF_CUDA(cudaMemsetAsync(r->d_labels, 0, sizeof(int32_t) * r->n, r->stream));
    }
    std::vector<int32_t> V((size_t)K * K);  // as phmrf_quantise hands V_i32 to the host cut
    smooth_costs_i32(ctx, V.data());
    if ((rc = swap_run(*r->cut, r->d_unary, r->d_edge_wi, V.data(), r->d_labels, n_iter, energy_out, energy_before_out,
                       r->stream)) != PHMRF_OK)
        return rc;
    if (labels_out) {
        PHMRF_CUDA(cudaMemcpyAsync(labels_out, r->d_labels, sizeof(int32_t) * r->n, cudaMemcpyDeviceToHost, r->stream));
        PHMRF_CUDA(cudaStreamSynchronize(r->stream));
    }
    r->have_labels = true;
    return PHMRF_OK;
}

// ---------------------------------------------------------------- next row (f-1)
int64_t phmrf_grid_edge_count(int kind, int64_t n1, int64_t n2, int num_neighbor) {
    if ((kind != 0 && kind != 1) || n1 < 1 || n2 < 1 || (num_neighbor != 8 && num_neighbor != 4)) return -1;
    if (kind == 1 && n1 != n2) return -1;
    return grid_edge_count(kind, n1, n2, num_neighbor);
}

int phmrf_grid_edges(int device, const double *X, int n_features, int kind, int64_t n1, int64_t n2, int num_neighbor,
                     double *edge_list_out, int64_t n_edges) {
    const int64_t expect = phmrf_grid_edge_count(kind, n1, n2, num_neighbor);
    if (!X || n_features < 1 || expect < 0 || n_edges != expect || (n_edges > 0 && !edge_list_out)) {
        set_error("phmrf_grid_edges: invalid arguments (kind 0/1, num_neighbor 8/4, n_edges from phmrf_grid_edge_count)");
        return PHMRF_E_INVALID;
    }
    int rc = use_device(device, "phmrf_grid_edges");
    if (rc) return rc;
    const int64_t n = kind == 1 ? n2 * (n2 + 1) / 2 : n1 * n2;
    DevBuf<double> dX, dE;
    if ((rc = dX.alloc(n * n_features)) || (rc = dE.alloc(3 * n_edges))) return rc;
    if (cudaMemcpy(dX, X, sizeof(double) * n * n_features, cudaMemcpyHostToDevice) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "upload X", __FILE__, __LINE__);
    if (n_edges > 0 && (rc = launch_grid_edges(dX, kind, n1, n2, num_neighbor, n_features, n, n_edges, dE, nullptr)))
        return rc;
    if (n_edges > 0 &&
        cudaMemcpy(edge_list_out, dE, sizeof(double) * 3 * n_edges, cudaMemcpyDeviceToHost) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "download edge list", __FILE__, __LINE__);
    return PHMRF_OK;
}

}  // extern "C"
