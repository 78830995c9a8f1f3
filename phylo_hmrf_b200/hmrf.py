"""``phyloHMRF`` -- the reference's model class re-hosted on the B200 library, hot path only.

Every method below keeps the name, argument order and return convention of the method it
replaces in the reference (file:line in each docstring), so code written against
``phylo_hmrf.py`` / ``base.py`` can call into this class unchanged for the per-region
E-step: emission -> integer cost arrays -> graph cut (host GCO) -> posteriors, cost
scalars and sufficient statistics.

The callers either side of the path (SURVEY 8 "next" rows) are re-hosted too: the fork-free EM
driver ``fit_accumulate_test`` (f-2) and, when the constructor is given the tree
(``edge_list``), the OU initialisation and SLSQP M-step of ``ou.py`` (f-3), which write
``means_`` / ``_covars_`` exactly where ``_do_mstep`` does (phylo_hmrf.py:1522-1524).  Without a
tree, ``means_`` / ``_covars_`` are plain attributes and ``init_fn`` / ``mstep_fn`` hooks can be
supplied by the caller.

There is no CPU fallback: all arithmetic of the hot path runs in ``libphmrf.so``.
"""
from __future__ import annotations

import numpy as np

from . import engine

small_eps = 1e-16  # phylo_hmrf.py:49


class _IncidentEdges:
    """List-of-lists view of ``_connected_edge`` (phylo_hmrf.py:674-689) backed by CSR
    arrays: ``inc[i]`` is the ascending list of edge indices incident to node ``i``."""

    def __init__(self, edge_ids, n_samples):
        e = np.asarray(edge_ids, dtype=np.int64).reshape(-1, 2)
        E = len(e)
        node = np.concatenate([e[:, 1], e[:, 0]]) if E else np.zeros(0, np.int64)
        eid = np.concatenate([np.arange(E), np.arange(E)]) if E else np.zeros(0, np.int64)
        order = np.lexsort((eid, node))
        self._eid = eid[order]
        self._off = np.zeros(n_samples + 1, dtype=np.int64)
        np.add.at(self._off, node + 1, 1)
        self._off = np.cumsum(self._off)
        self._n = n_samples

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        return self._eid[self._off[i]:self._off[i + 1]].tolist()


class phyloHMRF(object):
    """Hot-path subset of the reference's ``phyloHMRF(_BaseGraph)`` (phylo_hmrf.py:51-150)."""
    graph_cut = 'host'     # see __init__

    def __init__(self, n_samples, n_features, edge_list=None, branch_list=None, cons_param=1, beta=1.0, beta1=0.5,
                 initial_mode=0, initial_weight=0.3, initial_weight1=0.1, initial_magnitude=1, observation=None,
                 edge_list_1=None, len_vec=None, type_id=0, max_iter=10, n_components=1, run_id=0, estimate_type=0,
                 covariance_type='full', min_covar=1e-3, startprob_prior=1.0, transmat_prior=1.0, means_prior=0,
                 means_weight=0, covars_prior=1e-2, covars_weight=1, algorithm="viterbi", random_state=None,
                 n_iter=10, tol=1e-2, verbose=False, params="stmc", init_params="stmc", learning_rate=0.001,
                 device=0, implicit_grid=True, graph_cut='host'):
        if covariance_type != 'full':
            raise ValueError("the device path implements covariance_type='full' (phylo_hmrf.py:57)")
        if graph_cut not in ('host', 'device'):
            raise ValueError("graph_cut must be 'host' or 'device'")
        # 'host': the integer costs are downloaded and cut by csrc/gco.cpp, and last_quantise holds every integer
        # array.  'device': the same swap runs on the GPU on the region's own arrays (same labels), nothing but the
        # labels crosses PCIe, and last_quantise holds dwf and V_i32 only.  Costs the device cut does not run
        # (negative edge weights, non-submodular V) still go to the host.
        self.graph_cut = graph_cut
        self.n_components = int(n_components)
        self.n_features = int(n_features)
        self.n_samples = int(n_samples)
        self.run_id, self.estimate_type = run_id, int(estimate_type)
        self.covariance_type, self.min_covar = covariance_type, min_covar
        self.beta, self.beta1 = beta, beta1
        self.type_id, self.max_iter, self.n_iter, self.tol = type_id, max_iter, n_iter, tol
        self.lambda_0 = cons_param
        self.tree_edge_list, self.branch_params = edge_list, branch_list
        self.observation = observation
        self.edge_list_vec = edge_list_1
        self.len_vec = len_vec
        self.device = device
        self.implicit_grid = bool(implicit_grid)   # regions whose edge list IS the grid's take the implicit-grid kernels

        self._model = engine.Model(self.n_components, self.n_features, device)
        self._regions = []
        self._model_key = None

        self.initial_mode, self.initial_w1, self.initial_w1a, self.initial_w2 = (
            initial_mode, initial_weight, initial_weight1, initial_magnitude)
        self.init_fn = self.mstep_fn = self.finalize_fn = None
        if edge_list is not None:
            # OU tree algebra, initialisation and M-step (SURVEY 8 f-3; host side, phylo_hmrf.py:715-1528)
            from . import ou
            ou.attach(self, edge_list, initial_weight, initial_weight1, initial_magnitude, initial_mode, random_state)

        self.edge_potential = self._pairwise_potential()
        if observation is not None and len_vec is not None and edge_list_1 is not None:
            (self.edge_weightList_undirected_vec, self.edge_idList_undirected_vec,
             self.neighbor_edgeIdx_vec) = self._edge_weight_undirected_vec(observation, len_vec, edge_list_1)
            n_total = int(sum(int(v[0]) for v in len_vec))
            self.labels = np.zeros(n_total, dtype=np.int64)
            self.labels_local = np.zeros(n_total, dtype=np.int64)

    # ------------------------------------------------------------------ model upkeep
    def _sync_model(self):
        """Push means_/_covars_/edge_potential to the device when they changed."""
        key = (self.means_.tobytes(), self._covars_.tobytes(), self.edge_potential.tobytes())
        if key != self._model_key:
            self._model.set_model(self.means_, self._covars_, self.edge_potential)
            self._model_key = key

    @staticmethod
    def _where(a):
        """(address, shape, strides) of an array: two views with the same triple are the same memory."""
        a = np.asarray(a)
        return (a.__array_interface__['data'][0], a.shape, a.strides)

    def _region_for(self, X, edge_ids, edge_w, n=None):
        """The resident region built from these very edge arrays, else a temporary one.  A resident
        region computes from the features it was built from; when the caller passes other data
        (the reference uses the X it is given, phylo_hmrf.py:470-507) that data is uploaded first.
        X=None (with the node count n): the features play no part in what the caller computes."""
        n = len(X) if X is not None else int(n)
        for r, reg in enumerate(self._regions):
            if reg is not None and edge_ids is self.edge_idList_undirected_vec[r] and n == reg.n:
                if X is not None and self._where(X) != reg._x_where:
                    reg.update_X(np.asarray(X))
                    reg._x_where = self._where(X)
                    reg._host_logprob = None
                return reg, False
        reg = self._model.region(X if X is not None else np.zeros((n, self.n_features)), edge_ids, edge_w)
        reg._host_logprob = None
        return reg, True

    # ------------------------------------------------------------------ constants
    def _pairwise_potential(self):
        """phylo_hmrf.py:524-536: Potts ``beta*(1-I)``."""
        K = self.n_components
        V = np.full((K, K), float(self.beta))
        np.fill_diagonal(V, 0.0)
        self.edge_potential = V
        return V

    def _connected_edge(self, edge_list_1, n_samples):
        """phylo_hmrf.py:674-689."""
        return _IncidentEdges(edge_list_1, n_samples)

    def _edge_weight_undirected_vec(self, X, len_vec, edge_list_vec):
        """phylo_hmrf.py:567-598.  Also makes each region resident on the device."""
        num_region = len(len_vec)
        w_vec, id_vec, inc_vec = [None] * num_region, [None] * num_region, [None] * num_region
        for reg in self._regions:
            if reg is not None:
                reg.close()
        self._regions = []
        # under torchrun a rank keeps resident only the whole regions the plan gives it (row bands of
        # larger regions are made resident by the EM driver, _prepare_bands)
        from . import dist as _pdist, em as _em
        world, rank = _pdist.world_info()
        owned = set(_em.make_plan(len_vec, world)[0][rank]) if world > 1 else set(range(num_region))
        for r in range(num_region):
            n_samples, s1, s2 = int(len_vec[r][0]), int(len_vec[r][1]), int(len_vec[r][2])
            edge_list = np.asarray(edge_list_vec[r], dtype=np.float64)
            w = np.exp(-self.beta1 * edge_list[:, 2])
            ids = np.int64(edge_list[:, 0:2])
            w_vec[r], id_vec[r] = w, ids
            inc_vec[r] = self._connected_edge(ids, n_samples)
            if r not in owned:
                self._regions.append(None)
                continue
            reg = self._grid_region(np.asarray(X)[s1:s2], len_vec[r], ids, w) if getattr(self, "implicit_grid", True) else None
            if reg is None:
                reg = self._model.region(np.asarray(X)[s1:s2], ids, w)
            reg._x_where = self._where(np.asarray(X)[s1:s2])
            reg._host_logprob = None       # the host array the device log-likelihood currently equals
            self._regions.append(reg)
        return w_vec, id_vec, inc_vec

    def _grid_region(self, X, lv, ids, w, row0=0, row1=None, n_edges_region=None):
        """A region whose edge list is exactly what the reference's grid builders produce for its geometry
        (utility.py:1871-2053: len_vec carries kind, n1, n2; 8 or 4 neighbours; same ids in the same order;
        weights equal to 1e-12) is built on the device from that geometry: phase B then reads implicit
        neighbours and each edge weight once (64 instead of 160 bytes per node).  The host's own weights stay
        the source of the integer edge costs.  Anything else -> None (explicit neighbour slots).
        With row0/row1: the row band [row0,row1) of such a region; X holds the band's window (one halo row
        either side), ids/w the edges incident to the band's own nodes with window-local ids, and
        n_edges_region the edge count of the whole region."""
        from . import em, _lib
        geo = em._geometry(lv)
        if geo is None or len(ids) == 0:
            return None
        kind, n1, n2 = geo
        total = len(ids) if n_edges_region is None else int(n_edges_region)
        for nn in (8, 4):
            if int(_lib.lib().phmrf_grid_edge_count(kind, n1, n2, nn)) != total:
                continue
            reg = self._model.region_grid(X, kind, n1, n2, row0, row1, nn, float(self.beta1))
            gids, gw = reg.edges()
            if gids.shape == np.shape(ids) and np.array_equal(gids, ids) and np.allclose(gw, w, rtol=1e-12, atol=0.0):
                reg.set_edge_weights(w)
                return reg
            reg.close()
        return None

    # ------------------------------------------------------------------ phase A
    def _compute_log_likelihood(self, X):
        """phylo_hmrf.py:266-268 (sklearn 0.18 'full' density) on the device.  X that is the very slice a
        resident region was built from is not uploaded again."""
        self._sync_model()
        where = self._where(X)
        for reg in self._regions:
            if reg is not None and where == reg._x_where:
                reg.emit_loglik()
                reg._host_logprob = reg.logprob()
                return reg._host_logprob
        reg = self._model.region(X, np.zeros((0, 2), dtype=np.int64), np.zeros(0))
        try:
            reg.emit_loglik()
            return reg.logprob()
        finally:
            reg.close()

    def _device_cut(self, edge_w):
        """Whether graph_cut='device' applies to these costs (engine.swap_supported on the V_i32 the quantiser
        makes and the sign of the edge weights, both known on the host)."""
        if self.graph_cut != 'device':
            return False
        V_i32 = (np.asarray(self.edge_potential, dtype=np.float64) * self._model.quantiser()[2]).astype(np.int32)
        w = np.asarray(edge_w)
        return engine.swap_supported(V_i32, float(w.min()) if len(w) else 0.0)

    def _estimate_state_graphcuts_gco(self, X, init_labels1, edge_idList_undirected, edge_weightList_undirected,
                                      want_logprob=True, staged_labels=False):
        """phylo_hmrf.py:486-507: emission, integer cost arrays (GPU), alpha-beta swap with
        5000 cycles from ``init_labels1`` (host GCO, or the GPU with graph_cut='device').  Returns (labels, logprob)."""
        return self._graph_cut(X, init_labels1, edge_idList_undirected, edge_weightList_undirected, want_logprob,
                               staged_labels)[:2]

    def _graph_cut(self, X, init_labels1, edge_idList_undirected, edge_weightList_undirected, want_logprob=True,
                   staged_labels=False):
        """_estimate_state_graphcuts_gco -> (labels, logprob, the resident region that holds the labels on the
        device, or None)."""
        self._sync_model()
        reg, temp = self._region_for(X, edge_idList_undirected, edge_weightList_undirected)
        try:
            reg.emit_loglik()
            max_cycles1 = 5000
            on_device = self._device_cut(edge_weightList_undirected)
            if on_device:
                q = reg.quantise(want_unary=False, want_edges=False)
                labels = reg.graph_cut(init_labels1, n_iter=max_cycles1)
                self.last_quantise = dict(dwf=q["dwf"], V_i32=q["V_i32"])
            else:
                # resident regions keep page-locked staging buffers: the integer arrays go straight from the
                # device into the graph cut, and its labels straight back (no pageable copies in between)
                q = reg.quantise(staged=not temp)
                labels = engine.gco_cut_int(q["unary_i32"], edge_idList_undirected, q["w_i32"], q["V_i32"],
                                            n_iter=max_cycles1, algorithm='swap', init_labels=init_labels1,
                                            out=None if temp else reg.label_staging())
                self.last_quantise = q
                if not temp and not staged_labels:
                    labels = labels.copy()     # the staging buffer is overwritten by the region's next graph cut
            logprob = reg.logprob() if want_logprob else None
            reg._host_logprob = logprob
            return labels, logprob, reg if on_device and not temp else None
        finally:
            if temp:
                reg.close()

    def predict(self, X, region_id):
        """phylo_hmrf.py:470-484."""
        lv = self.len_vec[region_id]
        id1, id2 = int(lv[1]), int(lv[2])
        init_labels = self.labels_local[id1:id2].copy()
        state, logprob = self._estimate_state_graphcuts_gco(
            X, init_labels, self.edge_idList_undirected_vec[region_id], self.edge_weightList_undirected_vec[region_id])
        self.labels[id1:id2] = state
        return state, logprob

    # ------------------------------------------------------------------ phase B
    def _prepare_phase_b(self, reg, label, logprob):
        if logprob is not None and logprob is not reg._host_logprob:
            reg.set_logprob(logprob)
            reg._host_logprob = logprob
        reg.set_labels(np.asarray(label))

    def _pairwise_compare(self, label, neighbor_edgeIdx, edge_weightList, edge_idList):
        """phylo_hmrf.py:398-410 -> pp [N,K]."""
        self._sync_model()
        n = len(label)
        reg, temp = self._region_for(None, edge_idList, edge_weightList, n=n)
        try:
            if not reg.has_logp:
                reg.set_logprob(np.zeros((n, self.n_components)))   # the potential does not depend on it
                reg._host_logprob = None
            reg.set_labels(np.asarray(label))
            return reg.pairwise_potential(self.estimate_type)
        finally:
            if temp:
                reg.close()

    def _compute_posteriors_graph(self, X, label, logprob, region_id):
        """phylo_hmrf.py:334-355 -> (posteriors, pairwise_cost, pairwise_cost_normalize,
        unary_cost, cost1)."""
        self._sync_model()
        reg = self._regions[region_id]
        self._prepare_phase_b(reg, label, logprob)
        stats, sums, post = reg.estep_stats(self.estimate_type, want_post=True)
        self._last_stats = stats
        return (post,) + engine.costs_from_sums(sums, reg.n)

    def _compute_cost_v1(self, X, label, logprob1, pairwise_prob_normalize, neighbor_edgeIdx, edge_weightList,
                         edge_idList):
        """phylo_hmrf.py:374-396 -> (pairwise_cost, pairwise_cost_normalize, unary_cost, cost1).
        ``pairwise_prob_normalize`` is recomputed on the device from (label, edges): it is a
        function of exactly those inputs at the reference's only call site (:352)."""
        self._sync_model()
        reg, temp = self._region_for(None, edge_idList, edge_weightList, n=len(label))   # the costs do not read X
        try:
            reg.set_logprob(logprob1)
            reg._host_logprob = logprob1
            reg.set_labels(np.asarray(label))
            _, sums, _ = reg.estep_stats(self.estimate_type)
            return engine.costs_from_sums(sums, reg.n)
        finally:
            if temp:
                reg.close()

    def _pairwise_compare_ensemble(self, label, neighbor_edgeIdx, edge_weightList, edge_idList):
        """phylo_hmrf.py:438-447 -> mean over nodes of the label-pair potential."""
        n = len(label)
        return self._compute_cost_v1(np.zeros((n, self.n_features)), label, np.zeros((n, self.n_components)), None,
                                     neighbor_edgeIdx, edge_weightList, edge_idList)[0]

    def _predict_posteriors(self, X, len_vec, region_id, m_queue):
        """phylo_hmrf.py:297-322: one region of one EM iteration; puts
        ``(region_id, stats, labels, pairwise_cost, pairwise_cost_normalize, unary_cost,
        cost1)`` on ``m_queue``.  The log-likelihood and the posteriors stay on the device."""
        self._sync_model()
        lv = len_vec[region_id]
        s1, s2 = int(lv[1]), int(lv[2])
        reg = self._regions[region_id]
        init_labels = self.labels_local[s1:s2].copy()
        labels, _, resident = self._graph_cut(
            X[s1:s2], init_labels, self.edge_idList_undirected_vec[region_id],
            self.edge_weightList_undirected_vec[region_id], want_logprob=False, staged_labels=True)
        if resident is not reg:      # the device cut left its labels on the region already
            reg.set_labels(labels)
        stats, sums, _ = reg.estep_stats(self.estimate_type)
        c = engine.costs_from_sums(sums, reg.n)
        m_queue.put((region_id, stats, labels, c[0], c[1], c[2], c[3]))
        return True

    # ------------------------------------------------------------------ posterior summary
    def posterior_summary(self, region_id):
        """How confident the state map of a resident region is at each node, for the log-likelihood and labels
        it currently holds (after _predict_posteriors): dict of [N_r] arrays map_state (int32), map_prob,
        label_prob (posterior of the node's label) and entropy (nats); see phmrf_posterior_summary."""
        self._summary_launch(region_id)
        return self._summary_get(region_id)

    def _summary_launch(self, rid):
        self._regions[rid].posterior_summary(self.estimate_type)

    def _summary_get(self, rid):
        return self._regions[rid].get_posterior_summary()

    def _band_summary_launch(self, rid, bi):
        """The summary of one band's owned rows, for the band's current log-likelihood and label window."""
        self._bands[(rid, bi)][0].posterior_summary(self.estimate_type)

    def _band_summary_get(self, rid, bi):
        return self._bands[(rid, bi)][0].get_posterior_summary()

    # ------------------------------------------------------------------ statistics helpers
    def _initialize_sufficient_statistics(self):
        """base.py:562-569 + phylo_hmrf.py:691-698."""
        K, d = self.n_components, self.n_features
        return {'nobs': 0, 'start': np.zeros(K), 'trans': np.zeros((K, K)), 'post': np.zeros(K),
                'obs': np.zeros((K, d)), 'obs**2': np.zeros((K, d)), 'obs*obs.T': np.zeros((K, d, d))}

    def _accumulate_sufficient_statistics_1(self, stats, stats1):
        """base.py:571-580."""
        stats['post'] += stats1['post']
        stats['obs'] += stats1['obs']
        stats['obs*obs.T'] += stats1['obs*obs.T']
        return stats

    # ------------------------------------------------------------------ EM driver (SURVEY 8 f-2)
    def _init(self, X, lengths=None):
        """phylo_hmrf.py:205-264 (MiniBatchKMeans labels, per-cluster OU fit).  Out of the
        hot-path scope: supply `init_fn(model, X)` (it must set means_, _covars_, params_vec1,
        labels, labels_local) or subclass."""
        if getattr(self, "init_fn", None) is None:
            raise NotImplementedError("initialisation is outside the re-hosted hot path: set model.init_fn")
        self.init_fn(self, X)

    def _check(self):
        """base.py:515-538 / phylo_hmrf.py:152-182: parameter validation before fitting."""
        K, d = self.n_components, self.n_features
        self.means_ = np.asarray(self.means_)
        if self.means_.shape != (K, d):
            raise ValueError("means_ must have shape (n_components, n_features)")
        if np.asarray(self._covars_).shape != (K, d, d):
            raise ValueError("'full' covars must have shape (n_components, n_dim, n_dim)")

    def _do_mstep(self, stats):
        """phylo_hmrf.py:1500-1528 (K constrained SLSQP fits of the OU tree parameters).  Out of
        the hot-path scope: supply `mstep_fn(model, stats)` (it must update means_, _covars_
        and params_vec1) or subclass."""
        if getattr(self, "mstep_fn", None) is None:
            raise NotImplementedError("the OU M-step is outside the re-hosted hot path: set model.mstep_fn")
        self.stats = stats.copy()
        self.mstep_fn(self, stats)

    def _ou_param_varied_constraint(self, params_vec):
        """phylo_hmrf.py:985-1036: writes means_/_covars_ for the final parameters; delegated
        to `finalize_fn(model, params_vec)` when given."""
        if getattr(self, "finalize_fn", None) is not None:
            self.finalize_fn(self, params_vec)

    def fit_accumulate_test(self, X, len_vec, threshold, annotation, m_iter, lengths=None, n_threads=None,
                            posterior_summary=False):
        """base.py:301-455 without fork: see `phylo_hmrf_b200.em` (iteration, cost aggregation with the
        N_r/N weights, convergence tests, best-iteration bookkeeping; regions on a thread pool; under
        `torchrun` the regions -- or the row bands of a region too large for one GPU -- are spread over
        the ranks).  Returns (params_vec, params_vec1, params_vecList, iter_id1, iter_id2, cost_vec,
        t_labels).  posterior_summary=True also sets ``posterior_summary_``: the per-node summary of the
        posterior (map_state, map_prob, label_prob, entropy over all n_samples) at the iteration whose labels
        are t_labels."""
        from . import em
        return em.run(self, X, len_vec, threshold, annotation, m_iter, lengths=lengths, n_threads=n_threads,
                      posterior_summary=posterior_summary)

    # ------------------------------------------------------------------ row bands (SURVEY 8(e))
    def _prepare_bands(self, X, len_vec, banded, comm):
        """Make this rank's row bands resident: for each band the owned rows' features and the edges
        incident to them (ids local to the band's label window).  The rank that owns a banded region's
        graph cut also keeps an edge-only region for the integer edge weights of the whole region."""
        from . import em
        for entry in getattr(self, "_bands", {}).values():      # a second fit on the same model: start afresh
            entry[0].close()
        for reg in getattr(self, "_edge_regions", {}).values():
            reg.close()
        self._bands = {}
        self._edge_regions = {}
        X = np.asarray(X)
        for rid, plist in banded.items():
            lv = len_vec[rid]
            s1 = int(lv[1])
            kind, n1, n2 = em._geometry(lv)
            ids, w = self.edge_idList_undirected_vec[rid], self.edge_weightList_undirected_vec[rid]
            for bi, (rank, row0, row1) in enumerate(plist):
                if rank != comm.rank:
                    continue
                own0, own1, win0, win1 = em.band_window(kind, n1, n2, row0, row1)
                a, b = ids[:, 0], ids[:, 1]
                keep = ((a >= own0) & (a < own1)) | ((b >= own0) & (b < own1))
                reg = None
                if getattr(self, "implicit_grid", True):   # the band of a grid-built region: built on the device
                    reg = self._grid_region(X[s1 + win0:s1 + win1], lv, ids[keep] - win0, w[keep], row0, row1, len(ids))
                if reg is None:
                    reg = self._model.region(X[s1 + own0:s1 + own1], ids[keep] - win0, w[keep], n_window=win1 - win0,
                                             own_offset=own0 - win0)
                # every band quantises against the REGION's largest edge weight (pygco's down-weight factor)
                reg.set_weight_max(float(np.max(np.abs(w))) if len(w) else 0.0)
                self._bands[(rid, bi)] = (reg, own0, own1, win0, win1)
            if plist[0][0] == comm.rank:
                self._edge_regions[rid] = self._model.region(np.zeros((0, self.n_features)), ids, w,
                                                             n_window=int(lv[0]), own_offset=0)

    def _band_emit(self, rid, bi):
        """Emission of one band -> its max|logp|."""
        return self._bands[(rid, bi)][0].emit_loglik(want_absmax=True)

    def _band_quantise(self, rid, bi, dwf):
        """Integer unary [n_band, K] of one band under the region-wide down-weight factor."""
        return self._bands[(rid, bi)][0].quantise(dwf=dwf, want_edges=False, staged=True)["unary_i32"]

    def _region_edge_costs(self, rid, dwf):
        """(w_i32 [E], V_i32 [K,K]) of a whole banded region, on the rank that runs its graph cut."""
        reg = self._edge_regions[rid]
        reg.emit_loglik()
        q = reg.quantise(dwf=dwf, want_unary=False, staged=True)
        return q["w_i32"], q["V_i32"]

    def _band_estep(self, rid, bi, labels_window):
        """E-step of one band -> (statistics flattened post|obs|obs*obs.T, the three cost sums)."""
        reg = self._bands[(rid, bi)][0]
        reg.set_labels(labels_window)
        stats, sums, _ = reg.estep_stats(self.estimate_type)
        return np.concatenate([stats['post'].ravel(), stats['obs'].ravel(), stats['obs*obs.T'].ravel()]), sums

    def _banded_region(self, rid, len_vec, plist, comm):
        """One EM iteration of a region whose rows are spread over several ranks (called by every rank).
        -> (this rank's share of [statistics | 3 cost sums], the region's labels on the rank that ran
        the graph cut, else None)."""
        from . import em
        lv = len_vec[rid]
        n_region, s1, s2 = int(lv[0]), int(lv[1]), int(lv[2])
        kind, n1, n2 = em._geometry(lv)
        K = self.n_components
        owner = plist[0][0]
        mine = [bi for bi, (rank, _, _) in enumerate(plist) if rank == comm.rank]
        # emission; the region's max|logp| decides the down-weight factor every band must share
        absmax = comm.max(np.array([max([self._band_emit(rid, bi) for bi in mine] + [0.0])]))[0]
        w = self.edge_weightList_undirected_vec[rid]
        wv = (float(np.max(np.abs(w))) if len(w) else 0.0) * float(np.max(self.edge_potential))
        dwf = (wv if wv > absmax else absmax) + 1e-10          # pygco: max(max|unary|, max|w|*max V) + 1e-10
        # integer unary of every band to the owner of the graph cut
        unary = np.empty((n_region, K), dtype=np.int32) if comm.rank == owner else None
        for bi, (rank, row0, row1) in enumerate(plist):
            own0, own1, _, _ = em.band_window(kind, n1, n2, row0, row1)
            if rank == comm.rank:
                u = self._band_quantise(rid, bi, dwf)
                if comm.rank == owner:
                    unary[own0:own1] = u
                else:
                    comm.send(u, owner)
            elif comm.rank == owner:
                unary[own0:own1] = comm.recv((own1 - own0, K), np.int32, rank)
        labels = None
        if comm.rank == owner:
            w_i32, V_i32 = self._region_edge_costs(rid, dwf)
            if self._device_cut(w):
                labels = engine.gco_swap_device(unary, self.edge_idList_undirected_vec[rid], w_i32, V_i32, n_iter=5000,
                                                init_labels=self.labels_local[s1:s2].copy(), device=self.device)
            else:
                labels = engine.gco_cut_int(unary, self.edge_idList_undirected_vec[rid], w_i32, V_i32, n_iter=5000,
                                            algorithm='swap', init_labels=self.labels_local[s1:s2].copy())
        # label windows back to the bands, E-step per band
        n_stat = K * (1 + self.n_features + self.n_features * self.n_features)
        part = np.zeros(n_stat + 3)
        for bi, (rank, row0, row1) in enumerate(plist):
            _, _, win0, win1 = em.band_window(kind, n1, n2, row0, row1)
            if rank == comm.rank:
                lw = labels[win0:win1] if comm.rank == owner else comm.recv((win1 - win0,), np.int32, owner)
                flat, sums = self._band_estep(rid, bi, np.ascontiguousarray(lw, dtype=np.int32))
                part[:n_stat] += flat
                part[n_stat:] += sums
            elif comm.rank == owner:
                comm.send(np.ascontiguousarray(labels[win0:win1], dtype=np.int32), rank)
        return part, labels

    def close(self):
        for reg in self._regions:
            if reg is not None:
                reg.close()
        for entry in getattr(self, "_bands", {}).values():
            entry[0].close()
        for reg in getattr(self, "_edge_regions", {}).values():
            reg.close()
        self._regions, self._bands, self._edge_regions = [], {}, {}
        self._model.close()
