// SURVEY 8(f-1): the step immediately before the hot path -- the undirected 8-/4-neighbourhood
// edge list of a region with its edge distances, on the GPU.
//
// Reference: utility.py:1871-1973 edge_weightlist_grid3_undirected_unsym (diagonal region:
// row-major upper triangle incl. the diagonal, utility.py:2310-2317) and utility.py:1975-2053
// edge_weightlist_grid3_undirected (full n1 x n2 rectangle).  Forward directions right,
// lower-right, lower, lower-left (8) or right, lower (4) (utility.py:1898-1916), kept when
// the neighbour lies inside the region; d_ij = |xi-xj|^2 / (|xi||xj| + 1e-16), halved between
// two diagonal nodes of a diagonal region (utility.py:1919-1953); rows sorted by (id1,id2)
// (utility.py:1960), which for a dense region is: per node, neighbours in ascending id.
// Output format is the reference's: [E,3] float64 rows (id1, id2, d_ij).
#include <cub/cub.cuh>

#include "common.cuh"

namespace phmrf {

namespace {

struct Grid {
    int kind;  // 1 = diagonal region (upper triangle incl. diagonal), 0 = rectangle
    long long n1, n2;
    int nn;    // 8 or 4
};

__device__ __forceinline__ long long tri_start(long long B, long long x) { return x * B - (x * (x - 1)) / 2; }

// node id -> (x, y)
__device__ __forceinline__ void node_xy(const Grid &g, long long id, long long &x, long long &y) {
    if (g.kind == 0) {
        x = id / g.n2;
        y = id - x * g.n2;
    } else {
        const long long B = g.n2;
        // largest x with tri_start(x) <= id
        double bf = (double)B + 0.5;
        long long xx = (long long)(bf - sqrt(bf * bf - 2.0 * (double)id));
        if (xx < 0) xx = 0;
        if (xx > B - 1) xx = B - 1;
        while (xx > 0 && tri_start(B, xx) > id) --xx;
        while (xx < B - 1 && tri_start(B, xx + 1) <= id) ++xx;
        x = xx;
        y = xx + (id - tri_start(B, xx));
    }
}

__device__ __forceinline__ long long node_id(const Grid &g, long long x, long long y) {
    return g.kind == 0 ? x * g.n2 + y : tri_start(g.n2, x) + (y - x);
}

// the forward neighbours of (x,y) in ascending id order; returns how many are inside the region
__device__ __forceinline__ int forward_neighbours(const Grid &g, long long x, long long y, long long (&nid)[4],
                                                  bool (&both_diag)[4]) {
    int c = 0;
    const bool tri = g.kind != 0;
    const long long rows = tri ? g.n2 : g.n1, cols = g.n2;
    auto inside = [&](long long a, long long b) { return a >= 0 && a < rows && b >= 0 && b < cols && (!tri || a <= b); };
    // right
    if (inside(x, y + 1)) {
        nid[c] = node_id(g, x, y + 1);
        both_diag[c] = false;
        ++c;
    }
    if (g.nn == 8 && inside(x + 1, y - 1)) {  // lower left
        nid[c] = node_id(g, x + 1, y - 1);
        both_diag[c] = false;
        ++c;
    }
    if (inside(x + 1, y)) {  // lower
        nid[c] = node_id(g, x + 1, y);
        both_diag[c] = false;
        ++c;
    }
    if (g.nn == 8 && inside(x + 1, y + 1)) {  // lower right
        nid[c] = node_id(g, x + 1, y + 1);
        both_diag[c] = tri && x == y;
        ++c;
    }
    return c;
}

__global__ void grid_count_kernel(Grid g, long long n, int *__restrict__ counts) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        long long x, y, nid[4];
        bool bd[4];
        node_xy(g, i, x, y);
        counts[i] = forward_neighbours(g, x, y, nid, bd);
    }
}

__global__ void grid_fill_kernel(Grid g, long long n, int D, const double *__restrict__ X,
                                 const long long *__restrict__ offsets, double *__restrict__ edge_list) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        long long x, y, nid[4];
        bool bd[4];
        node_xy(g, i, x, y);
        const int c = forward_neighbours(g, x, y, nid, bd);
        const double *xi = X + i * D;
        double ni = 0.0;
        for (int j = 0; j < D; ++j) ni = fma(xi[j], xi[j], ni);
        ni = sqrt(ni);
        double *out = edge_list + offsets[i] * 3;
        for (int e = 0; e < c; ++e) {
            const double *xj = X + nid[e] * D;
            double nj = 0.0, dd = 0.0;
            for (int j = 0; j < D; ++j) {
                nj = fma(xj[j], xj[j], nj);
                const double t = xi[j] - xj[j];
                dd = fma(t, t, dd);
            }
            nj = sqrt(nj);
            double w = dd / (ni * nj + 1e-16);
            if (bd[e]) w *= 0.5;
            out[0] = (double)i;
            out[1] = (double)nid[e];
            out[2] = w;
            out += 3;
        }
    }
}

// ---- a row band of a region, built entirely on the device ------------------------------
struct Band {
    long long win_start, own_start, own_end;  // global node ids: window [win_start, ...), owned [own_start, own_end)
};

__device__ __forceinline__ double edge_distance(const double *xi, const double *xj, int D, bool halve) {
    double ni = 0.0, nj = 0.0, dd = 0.0;
    for (int j = 0; j < D; ++j) {
        ni = fma(xi[j], xi[j], ni);
        nj = fma(xj[j], xj[j], nj);
        const double t = xi[j] - xj[j];
        dd = fma(t, t, dd);
    }
    double w = dd / (sqrt(ni) * sqrt(nj) + 1e-16);
    return halve ? 0.5 * w : w;
}

__device__ __forceinline__ bool owned(const Band &b, long long id) { return id >= b.own_start && id < b.own_end; }

__global__ void band_count_kernel(Grid g, Band b, long long n_window, int *__restrict__ counts) {
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n_window;
         t += (long long)gridDim.x * blockDim.x) {
        const long long i = b.win_start + t;
        long long x, y, nid[4];
        bool bd[4];
        node_xy(g, i, x, y);
        const int c = forward_neighbours(g, x, y, nid, bd);
        int kept = 0;
        for (int e = 0; e < c; ++e) kept += (owned(b, i) || owned(b, nid[e])) ? 1 : 0;
        counts[t] = kept;
    }
}

// edge list of the band in (id1,id2) order: window-local ids, w = exp(-beta1 * d_ij)
__global__ void band_fill_kernel(Grid g, Band b, long long n_window, int D, const double *__restrict__ Xw,
                                 double beta1, const long long *__restrict__ offsets, long long *__restrict__ ids,
                                 double *__restrict__ w_out, unsigned long long *wmax_bits) {
    unsigned long long wmax = 0ull;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n_window;
         t += (long long)gridDim.x * blockDim.x) {
        const long long i = b.win_start + t;
        long long x, y, nid[4];
        bool bd[4];
        node_xy(g, i, x, y);
        const int c = forward_neighbours(g, x, y, nid, bd);
        long long pos = offsets[t];
        for (int e = 0; e < c; ++e) {
            if (owned(b, i) || owned(b, nid[e])) {
                const double w = exp(-beta1 * edge_distance(Xw + t * D, Xw + (nid[e] - b.win_start) * D, D, bd[e]));
                ids[2 * pos] = t;
                ids[2 * pos + 1] = nid[e] - b.win_start;
                w_out[pos] = w;
                const unsigned long long bits = (unsigned long long)__double_as_longlong(fabs(w));
                wmax = bits > wmax ? bits : wmax;
                ++pos;
            }
        }
    }
    if (wmax) atomicMax(wmax_bits, wmax);
}

// neighbour slots of every owned node in ascending neighbour id (the order in which the
// host builder meets the incident edges of a sorted edge list)
__global__ void band_ell_kernel(Grid g, Band b, long long n_own, long long ld, int D, const double *__restrict__ Xw,
                                double beta1, int W, int32_t *__restrict__ nbr_id, double *__restrict__ nbr_w) {
    const bool tri = g.kind != 0;
    const long long rows = tri ? g.n2 : g.n1, cols = g.n2;
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < n_own;
         o += (long long)gridDim.x * blockDim.x) {
        const long long i = b.own_start + o;
        long long x, y;
        node_xy(g, i, x, y);
        const double *xi = Xw + (i - b.win_start) * D;
        int s = 0;
        auto put = [&](long long a, long long c2) {
            if (a >= 0 && a < rows && c2 >= 0 && c2 < cols && (!tri || a <= c2)) {
                const long long j = node_id(g, a, c2);
                const bool halve = tri && x == y && a == c2;
                nbr_id[s * ld + o] = (int32_t)(j - b.win_start);
                nbr_w[s * ld + o] = exp(-beta1 * edge_distance(xi, Xw + (j - b.win_start) * D, D, halve));
                ++s;
            }
        };
        if (g.nn == 8) put(x - 1, y - 1);
        put(x - 1, y);
        if (g.nn == 8) put(x - 1, y + 1);
        put(x, y - 1);
        put(x, y + 1);
        if (g.nn == 8) put(x + 1, y - 1);
        put(x + 1, y);
        if (g.nn == 8) put(x + 1, y + 1);
        for (; s < W; ++s) {
            nbr_id[s * ld + o] = -1;
            nbr_w[s * ld + o] = 0.0;
        }
    }
}

// Forward-edge weights of every window node up to the last owned one, for the implicit-grid
// form of phase B: slot 0 = right, 1 = lower left, 2 = lower, 3 = lower right (ascending
// neighbour id); .x = w = exp(-beta1 * d_ij) (0 where the neighbour is outside the region),
// .y = the per-slot factor exp(beta * w), filled by fwd_factor_kernel.
__global__ void band_fwd_kernel(Grid g, Band b, long long n_fw, long long ldw, int D, const double *__restrict__ Xw,
                                double beta1, double2 *__restrict__ fwd) {
    const bool tri = g.kind != 0;
    const long long rows = tri ? g.n2 : g.n1, cols = g.n2;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n_fw;
         t += (long long)gridDim.x * blockDim.x) {
        const long long i = b.win_start + t;
        long long x, y;
        node_xy(g, i, x, y);
        const double *xi = Xw + t * D;
        auto put = [&](int slot, long long a2, long long c2, bool use) {
            double w = 0.0;
            if (use && a2 >= 0 && a2 < rows && c2 >= 0 && c2 < cols && (!tri || a2 <= c2)) {
                const long long j = node_id(g, a2, c2);
                const bool halve = tri && x == y && a2 == c2;
                w = exp(-beta1 * edge_distance(xi, Xw + (j - b.win_start) * D, D, halve));
            }
            fwd[slot * ldw + t] = make_double2(w, 1.0);
        };
        put(0, x, y + 1, true);
        put(1, x + 1, y - 1, g.nn == 8);
        put(2, x + 1, y, true);
        put(3, x + 1, y + 1, g.nn == 8);
    }
}

__global__ void fwd_factor_kernel(double2 *__restrict__ fwd, long long count, double beta, int weighted) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
        double2 v = fwd[i];
        v.y = exp(beta * (weighted ? v.x : 1.0));
        fwd[i] = v;
    }
}

}  // namespace

int launch_band_fwd(const double *Xw_dev, int kind, long long n1, long long n2, int nn, int D, long long win_start,
                    long long n_fw, double beta1, long long ldw, double2 *fwd, cudaStream_t s) {
    if (n_fw <= 0) return PHMRF_OK;
    Grid g{kind, n1, n2, nn};
    Band b{win_start, 0, 0};
    const int grid = (int)((n_fw + 255) / 256 < 148 * 16 ? (n_fw + 255) / 256 : 148 * 16);
    band_fwd_kernel<<<grid, 256, 0, s>>>(g, b, n_fw, ldw, D, Xw_dev, beta1, fwd);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

int launch_fwd_factor(double2 *fwd, long long count, double beta, int weighted, cudaStream_t s) {
    if (count <= 0) return PHMRF_OK;
    const long long blocks = (count + 255) / 256;
    fwd_factor_kernel<<<(int)(blocks < 2368 ? blocks : 2368), 256, 0, s>>>(fwd, count, beta, weighted);
    count_launch();
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

// Closed-form edge count of a dense region.
long long grid_edge_count(int kind, long long n1, long long n2, int nn) {
    if (kind == 0) {
        long long e = n1 * (n2 - 1) + (n1 - 1) * n2;  // right + lower
        if (nn == 8) e += 2 * (n1 - 1) * (n2 - 1);     // both diagonals
        return e;
    }
    const long long B = n2;
    long long e = B * (B - 1) / 2 /*right*/ + B * (B - 1) / 2 /*lower: (x+1,y), y>=x+1*/;
    if (nn == 8) e += B * (B - 1) / 2 /*lower right*/ + (B - 1) * (B - 2) / 2 /*lower left: y-1>=x+1*/;
    return e;
}

int launch_grid_edges(const double *X_dev, int kind, long long n1, long long n2, int nn, int D, long long n,
                      long long n_edges, double *edge_list_dev, cudaStream_t s) {
    Grid g{kind, n1, n2, nn};
    DevBuf<int> counts;
    DevBuf<long long> offsets;
    DevBuf<unsigned char> tmp;
    size_t tmp_bytes = 0;
    int rc;
    if ((rc = counts.alloc(n + 1)) || (rc = offsets.alloc(n + 1))) return rc;
    const int grid = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
    grid_count_kernel<<<grid, 256, 0, s>>>(g, n, counts);
    count_launch();
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts.get(), offsets.get(), n, s);
    if ((rc = tmp.alloc((int64_t)tmp_bytes))) return rc;
    cub::DeviceScan::ExclusiveSum(tmp.get(), tmp_bytes, counts.get(), offsets.get(), n, s);
    count_launch();
    grid_fill_kernel<<<grid, 256, 0, s>>>(g, n, D, X_dev, offsets, edge_list_dev);
    count_launch();
    cudaError_t e = cudaStreamSynchronize(s);
    (void)n_edges;
    if (e != cudaSuccess) return cuda_fail(e, "grid edge kernels", __FILE__, __LINE__);
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

long long grid_row_start(int kind, long long n1, long long n2, long long row) {
    (void)n1;
    return kind == 0 ? row * n2 : row * n2 - (row * (row - 1)) / 2;
}

// Builds, for the band of rows [row0,row1) of a region whose window features Xw_dev ([n_window,D],
// row-major) are on the device: the edge list (ids window-local, weights), and the ELL slots.
// ids_dev / w_dev may be nullptr for a counting call (returns the edge count in *n_edges).
int launch_band_graph(const double *Xw_dev, int kind, long long n1, long long n2, int nn, int D, long long win_start,
                      long long own_start, long long own_end, long long n_window, double beta1, long long ld,
                      int32_t *nbr_id, double *nbr_w, long long *ids_dev, double *w_dev, long long *n_edges,
                      unsigned long long *wmax_bits, cudaStream_t s) {
    Grid g{kind, n1, n2, nn};
    Band b{win_start, own_start, own_end};
    const long long n_own = own_end - own_start;
    const int grid = (int)((n_window + 255) / 256 < 148 * 16 ? (n_window + 255) / 256 : 148 * 16);
    // both calls: the edges each window node starts, and their exclusive scan (the first edge of each node)
    DevBuf<int> counts;
    DevBuf<long long> offsets;
    DevBuf<unsigned char> tmp;
    size_t tmp_bytes = 0;
    int rc;
    if ((rc = counts.alloc(n_window + 1)) || (rc = offsets.alloc(n_window + 1))) return rc;
    PHMRF_CUDA(cudaMemsetAsync(counts, 0, sizeof(int) * (n_window + 1), s));
    band_count_kernel<<<grid, 256, 0, s>>>(g, b, n_window, counts);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts.get(), offsets.get(), n_window + 1, s);
    if ((rc = tmp.alloc((int64_t)tmp_bytes))) return rc;
    cub::DeviceScan::ExclusiveSum(tmp.get(), tmp_bytes, counts.get(), offsets.get(), n_window + 1, s);
    if (ids_dev == nullptr) {
        count_launch(2);
        long long total = 0;
        PHMRF_CUDA(cudaMemcpyAsync(&total, offsets + n_window, sizeof(long long), cudaMemcpyDeviceToHost, s));
        PHMRF_CUDA(cudaStreamSynchronize(s));
        *n_edges = total;
        return PHMRF_OK;
    }
    PHMRF_CUDA(cudaMemsetAsync(wmax_bits, 0, sizeof(unsigned long long), s));
    band_fill_kernel<<<grid, 256, 0, s>>>(g, b, n_window, D, Xw_dev, beta1, offsets, ids_dev, w_dev, wmax_bits);
    if (n_own > 0) {
        const int grid2 = (int)((n_own + 255) / 256 < 148 * 16 ? (n_own + 255) / 256 : 148 * 16);
        band_ell_kernel<<<grid2, 256, 0, s>>>(g, b, n_own, ld, D, Xw_dev, beta1, nn, nbr_id, nbr_w);
    }
    count_launch(4);
    cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return cuda_fail(e, "band graph kernels", __FILE__, __LINE__);
    PHMRF_CUDA(cudaGetLastError());
    return PHMRF_OK;
}

}  // namespace phmrf
