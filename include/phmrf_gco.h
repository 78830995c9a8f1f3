/*
 * phmrf_gco.h -- C ABI of the host graph-cut step (libphmrf_gco.so).
 *
 * Replaces pygco.cut_general_graph (phylo_hmrf.py:496-498) on integer costs: the general-graph
 * alpha-beta swap / alpha-expansion of GCO v3.0 (GCoptimizationGeneralGraph with setDataCost,
 * setNeighbors per edge, setSmoothCost, setLabel per site, swap(n_iter) / expansion(n_iter)),
 * implemented in csrc/gco.cpp with the same move order, stopping rule and cut (see there).
 * The graph cut stays on the host; it consumes the integer arrays produced on the GPU
 * by phmrf_quantise.  No state outlives a call; errors are reported through the return
 * code / phmrf_gco_last_error().
 */
#ifndef PHMRF_GCO_H_
#define PHMRF_GCO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { PHMRF_GCO_SWAP = 0, PHMRF_GCO_EXPANSION = 1 };

/* unary [n_sites*n_labels] (site-major, GCoptimization.h:337), edge_ids [n_edges*2] with
 * id1<id2, edge_w [n_edges], smooth [n_labels*n_labels], init_labels [n_sites] or NULL,
 * labels_out [n_sites].  energy_out (nullable) receives the final total energy and
 * energy_before_out (nullable) the energy of the initial labelling.  n_iter: cycles at most,
 * -1 for no limit (for expansion this is plain cycles, not GCO's adaptive ones).
 * Returns 0, or -1 on invalid arguments / a GCO exception. */
int phmrf_gco_cut_general_graph(int64_t n_sites, int32_t n_labels, const int32_t *unary, const int64_t *edge_ids,
                                const int32_t *edge_w, int64_t n_edges, const int32_t *smooth,
                                const int32_t *init_labels, int32_t n_iter, int32_t algorithm,
                                int32_t *labels_out, long long *energy_out, long long *energy_before_out);

const char *phmrf_gco_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* PHMRF_GCO_H_ */
