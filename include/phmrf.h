/*
 * phmrf.h -- C ABI of the B200-native Phylo-HMRF E-step hot path (libphmrf.so).
 *
 * The reference (ma-compbio/Phylo-HMRF) has no FFI of its own: its boundary is a set of
 * Python methods plus two third-party callables.  Each entry point below names the
 * reference interface it replaces (file:line relative to the reference tree).
 *
 * Conventions
 *   - plain pointers and sizes only; every host buffer is owned by the caller and is not
 *     referenced after the call returns; device memory lives behind the opaque handles.
 *   - all entry points return 0 on success and a negative PHMRF_E_* code on failure and
 *     never call exit()/throw across the ABI; phmrf_last_error() gives the message of the
 *     last failure on the calling thread.
 *   - handles are not thread-safe; distinct regions may be driven from distinct threads.
 *   - [N,K] host arrays are C-order (row = node), exactly as the reference's NumPy arrays.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     PHMRF_E_CUDA.
 */
#ifndef PHMRF_H_
#define PHMRF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHMRF_ABI_VERSION 1

enum {
    PHMRF_OK = 0,
    PHMRF_E_INVALID = -1,     /* bad argument (shape, null pointer, id out of range)            */
    PHMRF_E_CUDA = -2,        /* CUDA runtime error / no device                                 */
    PHMRF_E_NOT_SPD = -3,     /* covariance not symmetric positive-definite (reference raises
                                 ValueError via sklearn 0.18 gmm.py / base.py:526-538)          */
    PHMRF_E_STATE = -4,       /* call order violated (e.g. quantise before emit)                */
    PHMRF_E_UNSUPPORTED = -5  /* shape outside the compiled kernel range                        */
};

typedef struct phmrf_ctx phmrf_ctx;       /* one model (K states, d leaves) on one device        */
typedef struct phmrf_region phmrf_region; /* one synteny region, or one row band of a region     */

int phmrf_abi_version(void);
const char *phmrf_last_error(void);

/* ------------------------------------------------------------------ model ------------- */

/* Replaces the state the hot path reads from the model object: means_ [K,d], _covars_
 * [K,d,d] (phylo_hmrf.py:1521-1524) and edge_potential [K,K] (phylo_hmrf.py:99,524-536). */
int phmrf_ctx_create(int device, int n_states, int n_features, phmrf_ctx **out);
int phmrf_ctx_destroy(phmrf_ctx *ctx);

/* Host side of sklearn-0.18 _log_multivariate_normal_density_full (behind
 * phylo_hmrf.py:266-268): per-state lower Cholesky (retry with +1e-7*I, else
 * PHMRF_E_NOT_SPD), log-det, and the inverse factor the kernels consume.  V is the label
 * compatibility matrix handed to pygco (phylo_hmrf.py:495); the Potts form beta*(1-I)
 * produced by _pairwise_potential takes the fast path, any other V the general one. */
int phmrf_set_model(phmrf_ctx *ctx, const double *means, const double *covars, const double *V);

/* The three scale factors of pygco's float -> int conversion (yujiali/pygco pygco.py, behind
 * phylo_hmrf.py:496-498): _UNARY_FLOAT_PRECISION = 1e5 for the unary costs,
 * _PAIRWISE_FLOAT_PRECISION = 1e3 for the edge weights and _SMOOTH_COST_PRECISION = 1e2 for the
 * label compatibility matrix V (pygco's own rule: "pairwise * smooth = unary", 1e3 * 1e2 = 1e5,
 * so that w_ij * V[a,b] lands on the unary's scale).  These are the defaults; the setter exists
 * because pygco is not vendored by the reference and is unpinned (README.md:84), so a maintainer
 * can match whatever their installed pygco uses (INTEGRATION.md shows how to check). */
int phmrf_set_quantiser(phmrf_ctx *ctx, double unary_precision, double pairwise_precision, double smooth_precision);
int phmrf_get_quantiser(const phmrf_ctx *ctx, double *unary_precision, double *pairwise_precision,
                        double *smooth_precision);

/* ------------------------------------------------------------------ host staging ------ */

/* Page-locked host memory for the arrays that cross PCIe every EM iteration of a region: the
 * integer unary / edge weights pygco hands to the graph cut (phylo_hmrf.py:496-498; device ->
 * host) and the labels it returns (host -> device).  The reference holds these as ordinary NumPy
 * arrays (pageable); copies to or from pageable memory are staged by the driver and serialise,
 * copies to or from these buffers run at the link rate and overlap with kernels and with copies in
 * the other direction.  Any entry point accepts either kind of pointer. */
int phmrf_host_alloc(int64_t bytes, void **out);
int phmrf_host_free(void *p);

/* ------------------------------------------------------------------ region ------------ */

/* Replaces the per-region inputs of _predict_posteriors (phylo_hmrf.py:297-322): X[s1:s2]
 * and the output of _edge_weight_undirected_vec / _connected_edge (phylo_hmrf.py:567-598,
 * 674-689): edge_ids [E,2] (int64, id1<id2, sorted by (id1,id2)) and edge weights
 * w = exp(-beta1*d_ij) [E].
 *
 * Row-band sharding: a band owns nodes [own_offset, own_offset+n_own) of a label window of
 * n_window nodes; edge ids are window-local and every edge incident to an owned node must
 * be present (edges between two non-owned nodes are ignored).  A whole region is the
 * special case own_offset=0, n_own=n_window.  X holds the n_own owned rows.
 * stream: a cudaStream_t to enqueue on (e.g. torch.cuda.Stream.cuda_stream) or NULL for a
 * stream owned by the region. */
int phmrf_region_create(phmrf_ctx *ctx, const double *X, int64_t n_own, int64_t n_window, int64_t own_offset,
                        const int64_t *edge_ids, const double *edge_w, int64_t n_edges, void *stream,
                        phmrf_region **out);
/* Re-upload the owned rows of X [n_own,d] into a resident region (the `X[s1:s2]` argument
 * of _predict_posteriors, phylo_hmrf.py:297-303, when the caller passes it every
 * iteration).  Enqueued on the region's stream; X must stay valid until the next sync. */
int phmrf_region_update_X(phmrf_region *r, const double *X);
int phmrf_region_destroy(phmrf_region *r);
int phmrf_region_sync(phmrf_region *r);
int64_t phmrf_region_device_bytes(const phmrf_region *r);

/* ------------------------------------------------------------------ phase A ----------- */

/* _compute_log_likelihood (phylo_hmrf.py:266-268, called at :489): enqueue the emission
 * kernel; the [K,N] log-likelihood stays on the device.  absmax_out (nullable) receives
 * max|logp| over the owned nodes (the data term of pygco's down_weight_factor); asking for
 * it synchronises the region's stream. */
int phmrf_emit_loglik(phmrf_region *r, double *absmax_out);

/* Copy the log-likelihood to a host [n_own,K] array (return value of
 * _compute_log_likelihood / second return of _estimate_state_graphcuts_gco). */
int phmrf_get_logprob(phmrf_region *r, double *logprob_out);

/* Replace the resident log-likelihood by a caller-supplied [n_own,K] array: the `logprob`
 * argument of _compute_posteriors_graph / _compute_cost_v1 (phylo_hmrf.py:334, 374) when
 * it is not the array the emission kernel just produced. */
int phmrf_set_logprob(phmrf_region *r, const double *logprob);

/* The float->int conversion inside pygco.cut_general_graph (yujiali/pygco, called at
 * phylo_hmrf.py:496-498 with down_weight_factor=None):
 *   dwf = max(max|unary|, max|w|*max(V)) + 1e-10
 *   unary_i32 = trunc((-logp/dwf)*1e5); w_i32 = trunc((w/dwf)*1e3); V_i32 = trunc(V*1e2)
 * (scale factors: phmrf_set_quantiser)
 * dwf_in > 0 overrides the region-local value (bands of one region must share the
 * all-reduced maximum).  Any output pointer may be NULL (the integer unary then stays on
 * the device for phmrf_labels_argmin_unary).  Entries whose scaled value lies within
 * relative `tol` of a truncation boundary are reported: flat indices (node*K+state) go to
 * boundary_idx (capacity boundary_cap), their total count to n_boundary. */
int phmrf_quantise(phmrf_region *r, double dwf_in, double tol, int32_t *unary_i32_out, int32_t *w_i32_out,
                   int32_t *V_i32_out, double *dwf_out, int64_t *boundary_idx, int64_t boundary_cap,
                   int64_t *n_boundary);

/* ------------------------------------------------------------------ phase B ----------- */

/* Labels of the whole window (owned nodes + halo), as returned by the graph cut
 * (phylo_hmrf.py:496-498) -- int32, values in [0,K). */
int phmrf_set_labels(phmrf_region *r, const int32_t *labels_window);

/* Bench / test stand-in for the graph cut (SURVEY 8(d)): labels = arg-min_k of the device
 * integer unary (first minimum).  Only valid for whole regions (n_own == n_window). */
int phmrf_labels_argmin_unary(phmrf_region *r, int32_t *labels_out);

/* _compute_posteriors_graph + _compute_cost_v1 + the statistics triple
 * (phylo_hmrf.py:334-355, 374-468, 311-314) in one fused pass over the owned nodes:
 *   stats_out [K*(1+d+d*d)] = post[K] | obs[K,d] | obs*obs.T[K,d,d]
 *   cost_sums_out [3] = sum_i sum_{e in inc(i)} V[l_nbr,l_i]*w_e ; sum_i ln(pwn[i,l_i]+1e-16) ;
 *                       sum_i logp[i,l_i]          (un-normalised, so that bands add up)
 * post_out (nullable) receives the posteriors [n_own,K].  estimate_type==3 weights the
 * pairwise term by w (phylo_hmrf.py:431-434, 460-462).  The results also stay in a device
 * buffer of K*(1+d+d*d)+3 doubles (phmrf_stats_device_ptr) for an NCCL all-reduce. */
int phmrf_estep_stats(phmrf_region *r, int estimate_type, double *post_out, double *stats_out,
                      double *cost_sums_out);
/* _pairwise_compare (phylo_hmrf.py:398-410): the neighbour-weighted pairwise potential
 * pp [n_own,K] for the current labels.  The fused E-step never materialises it; this entry
 * point exists for signature parity and for tests. */
int phmrf_pairwise_potential(phmrf_region *r, int estimate_type, double *pp_out);
void *phmrf_stats_device_ptr(phmrf_region *r);
/* Row bands of ONE region spread over several GPUs must share pygco's down_weight_factor.
 * phmrf_absmax_device_ptr: device address of max|logp| of this band, stored as the uint64 bit
 * pattern of a non-negative double (integer order == numeric order), ready for an NCCL
 * max-all-reduce between phmrf_emit_loglik_async and phmrf_quantise_async.
 * phmrf_region_set_weight_max: replace the band-local max|w| by the region-wide one. */
void *phmrf_absmax_device_ptr(phmrf_region *r);
int phmrf_region_set_weight_max(phmrf_region *r, double wmax);
double phmrf_region_weight_max(const phmrf_region *r);
int64_t phmrf_stats_len(const phmrf_ctx *ctx);

/* Enqueue-only forms used by the bench (no host copies, no synchronisation). */
int phmrf_emit_loglik_async(phmrf_region *r);
int phmrf_quantise_async(phmrf_region *r, double dwf_in, double tol);
int phmrf_estep_stats_async(phmrf_region *r, int estimate_type);

/* Number of kernel launches this library has enqueued so far (bench "gpu_launches"). */
int64_t phmrf_launch_count(void);

/* ------------------------------------------------------------------ graph cut ----------- */

/* The alpha-beta swap of csrc/gco.cpp (phmrf_gco_cut_general_graph with algorithm PHMRF_GCO_SWAP) on the
 * device, host arrays in, with the same meaning.  Same labels and energies as the host cut: every move takes
 * the smallest sink side of all minimum cuts, which depends on the energy alone.  Sites are indexed with 64
 * bits (no n_sites*n_labels < 2^31 limit).  Errors where the host returns one (a term above
 * GCO_MAX_ENERGYTERM in an executed move, a bad init label, edges not 0 <= id1 < id2 < n_sites);
 * PHMRF_E_UNSUPPORTED for a negative edge weight or V[a][b] + V[b][a] < V[a][a] + V[b][b] (non-submodular
 * moves, which only the host cut runs). */
int phmrf_graph_cut_swap(int device, int64_t n_sites, int32_t n_labels, const int32_t *unary, const int64_t *edge_ids,
                         const int32_t *edge_w, int64_t n_edges, const int32_t *smooth, const int32_t *init_labels,
                         int32_t n_iter, int32_t *labels_out, long long *energy_out, long long *energy_before_out);
/* The same on a whole region's own integer arrays from the last phmrf_quantise (unary, edge weights and V_i32):
 * nothing crosses PCIe but the init labels (NULL: all 0) and, if labels_out != NULL, the result.  The labels
 * stay resident for phmrf_estep_stats.  A band (n_own != n_window) is PHMRF_E_INVALID.  The region's cut scratch
 * is allocated at its first call and counted in phmrf_region_device_bytes. */
int phmrf_region_graph_cut(phmrf_region *r, const int32_t *init_labels, int32_t n_iter, int32_t *labels_out,
                           long long *energy_out, long long *energy_before_out);

/* ------------------------------------------------------------------ next row (f-1) ---- */

/* utility.py:1871-1973 (edge_weightlist_grid3_undirected_unsym, kind=1: diagonal region of
 * n2 bins, row-major upper triangle incl. the diagonal) and utility.py:1975-2053
 * (edge_weightlist_grid3_undirected, kind=0: n1 x n2 rectangle): the undirected 8- or
 * 4-neighbourhood edge list of a DENSE region with d_ij = |xi-xj|^2/(|xi||xj|+1e-16) (halved
 * between two diagonal nodes), sorted by (id1,id2), in the reference's [E,3] float64 format
 * (id1, id2, d_ij).  X is the host [n,d] feature matrix in the region's node order.
 * phmrf_grid_edge_count gives E (closed form) so the caller can size edge_list_out. */
int64_t phmrf_grid_edge_count(int kind, int64_t n1, int64_t n2, int num_neighbor);
int phmrf_grid_edges(int device, const double *X, int n_features, int kind, int64_t n1, int64_t n2, int num_neighbor,
                     double *edge_list_out, int64_t n_edges);

/* A region -- or the row band [row0,row1) of one -- built entirely on the device from the
 * grid geometry: X_window holds the features of rows [max(row0-1,0), min(row1+1,rows)) in the
 * region's node order; the 8-/4-neighbour graph, d_ij, w = exp(-beta1*d_ij) (phylo_hmrf.py:585)
 * and the neighbour slots are computed by kernels, so no edge array crosses PCIe.  The edge list
 * (window-local ids, sorted by (id1,id2); every edge incident to an owned node) can be read back
 * for the host graph cut with phmrf_region_edges. */
int phmrf_region_create_grid(phmrf_ctx *ctx, const double *X_window, int kind, int64_t n1, int64_t n2, int64_t row0,
                             int64_t row1, int num_neighbor, double beta1, void *stream, phmrf_region **out);
int64_t phmrf_region_n_edges(const phmrf_region *r);
int64_t phmrf_region_n_own(const phmrf_region *r);
int64_t phmrf_region_n_window(const phmrf_region *r);
int64_t phmrf_region_own_offset(const phmrf_region *r);
int phmrf_region_edges(phmrf_region *r, int64_t *edge_ids_out, double *edge_w_out);

/* For a region built by phmrf_region_create_grid whose edge list the caller ALSO holds as the reference's
 * host arrays (output of _edge_weight_undirected_vec, phylo_hmrf.py:567-598): hand over the host's
 * w = exp(-beta1*d_ij) [E] (same order as phmrf_region_edges).  The integer conversion of the edge weights
 * (phmrf_quantise) and max|w| then use exactly these values -- NumPy's exp and the device's may differ in
 * the last bit, and the integer arrays handed to the graph cut must be those pygco would build from the
 * host array -- while phase B keeps the device-built weights of the implicit grid. */
int phmrf_region_set_edge_weights(phmrf_region *r, const double *edge_w, int64_t n_edges);

/* ------------------------------------------------------------------ preprocessing ----- */

/* Per-species rescale to a common range followed by the log transform (utility.py:867-897
 * normalize_feature, utility.py:362 x = log(1 + x1)).  x is [n,d] row-major on the host and is
 * transformed in place: negatives are clamped to 0, column i is mapped linearly from its own
 * [min_i, max_i] to [x_min, x_max]; a negative *x_min / *x_max selects the median of the column
 * minima / maxima and the value used is written back.  colminmax_out is [d,2].  log1p != 0
 * applies log(1 + x) afterwards. */
int phmrf_prep_normalise(int device, double *x, int64_t n, int d, double *x_min, double *x_max, double *colminmax_out,
                         int log1p);

/* One region's contact image and its node features (utility.py:1519-1598
 * write_matrix_image_Ctrl_unsym1 for kind 1, :1704-1783 write_matrix_image_Ctrl_sym1 for kind 0,
 * without the edge list -- phmrf_grid_edges / phmrf_region_create_grid build that):
 *   1. scatter the n bin pairs value[i,:] at (pos[i,0]-start1, pos[i,1]-start2) into an n1 x n2 x d
 *      image (kind 1: n1 == n2, start1 == start2, written symmetrically; utility.py:2192-2226,
 *      2332-2365).  A pair listed twice keeps one of its values, unspecified which (the
 *      reference keeps the last);
 *   2. per species, the 3x3 median hole fill in the reference's sequential raster order
 *      (utility.py:603-659; executed as a 2i+j wavefront, which preserves every dependency);
 *   3. filter_mode 0: Perona-Malik anisotropic diffusion, niter steps, conduction
 *      exp(-(delta/kappa)^2), step gamma, float32 like medpy's implementation (the call at
 *      utility.py:1566-1573); filter_mode 2 with sigma > 0: scipy.ndimage.gaussian_filter(plane, sigma)
 *      (float64, mode 'reflect', truncate 4; utility.py:1585-1589); any other combination: no filter
 *      (filter_mode 1, the skimage bilateral filter, is not built);
 *   4. nodes in the reference's order: the upper triangle row by row (kind 1) or the whole block
 *      (kind 0) -> data_out [n_nodes, d] row-major (utility.py:2295-2329, 2368-2400).
 * image_out (nullable) receives the filtered image [n1, n2, d]. */
int phmrf_prep_region_image(int device, const double *value, const int64_t *pos, int64_t n, int d, int kind,
                            int64_t start1, int64_t start2, int64_t n1, int64_t n2, int filter_mode, int niter,
                            double kappa, double gamma, double sigma, double *data_out, double *image_out);


#ifdef __cplusplus
}
#endif
#endif /* PHMRF_H_ */
