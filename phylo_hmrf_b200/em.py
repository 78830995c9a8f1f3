"""EM driver of the re-hosted model (SURVEY 8 f-2): what `fit_accumulate_test` (base.py:301-455)
does, organised as three pieces.

* :class:`CostHistory` -- the convergence tests and the best-iteration bookkeeping
  (base.py:319, 402-435).
* :class:`Comm` -- the exchanges between the processes of a `torchrun` launch (one per GPU).  The
  reference forks one process per region and sums what comes back on a queue (base.py:357-396);
  here every rank works on the pieces `dist.plan_shards` gives it -- whole regions, or row bands of
  a region too large for one GPU -- and the per-region totals are combined with ONE all-reduce per
  iteration.  Initialisation and M-step run on rank 0 and the parameters are broadcast, so the
  ranks cannot drift apart (k-means and SLSQP are not bit-reproducible across processes).
* :func:`run` -- the iteration itself.

A banded region goes through the same arithmetic as a whole one: emission per band, max|logp|
max-reduced so that every band quantises with the region's down-weight factor, the integer unary
gathered on the region's owner for the (host, single-process) graph cut, label windows (band + one
halo row either side) sent back, E-step per band, statistics and cost sums added up.
"""
from __future__ import annotations

import queue as _queue
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import dist as pdist
from .engine import costs_from_sums


class CostHistory(object):
    """Relative-change stop rule and best-so-far bookkeeping of base.py:319, 402-435."""

    def __init__(self, threshold, patience=50):
        self.threshold = threshold
        self.patience = patience            # iterations allowed after the best cost (counted from iteration 3 on)
        self.previous = (0.001, 0.001, 0.001)   # pairwise, unary, total
        self.rows = []
        self.best = (0, 1000)               # lowest total cost so far: (iteration, cost)
        self.best_settled = (0, 1000)       # the same, iterations 0-2 ignored

    def add(self, it, pairwise, unary, total):
        """-> (new overall best?, new settled best?, stop?)"""
        change = [abs((now - before) * 1.0 / before) for now, before in zip((pairwise, unary, total), self.previous)]
        self.previous = (pairwise, unary, total)
        self.rows.append([it, pairwise, unary, total])
        is_best = total < self.best[1]
        if is_best:
            self.best = (it, total)
        is_settled = total < self.best_settled[1] and it >= 3
        if is_settled:
            self.best_settled = (it, total)
        flat = (change[0] < self.threshold and change[1] < self.threshold) or change[2] < self.threshold
        stop = (flat and it > 5) or (it - self.best_settled[0] > self.patience)
        return is_best, is_settled, stop


class Comm(object):
    """torch.distributed as NumPy-in / NumPy-out; every method is the identity in a single process."""

    def __init__(self):
        self.size, self.rank = pdist.world_info()
        if self.size > 1:
            import torch
            import torch.distributed as td
            self.torch, self.td = torch, td
            self.where = "cuda" if td.get_backend() == "nccl" else "cpu"

    def _t(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.where)

    def sum(self, a):
        if self.size == 1:
            return a
        t = self._t(a)
        self.td.all_reduce(t)
        return t.cpu().numpy()

    def max(self, a):
        if self.size == 1:
            return a
        t = self._t(a)
        self.td.all_reduce(t, op=self.td.ReduceOp.MAX)
        return t.cpu().numpy()

    def send(self, a, dst):
        self.td.send(self._t(a), dst)

    def recv(self, shape, dtype, src):
        t = self.torch.empty(tuple(shape), dtype=getattr(self.torch, np.dtype(dtype).name), device=self.where)
        self.td.recv(t, src)
        return t.cpu().numpy()

    def broadcast_array(self, a, src):
        if self.size == 1:
            return a
        t = self._t(a)
        self.td.broadcast(t, src)
        return t.cpu().numpy()

    def broadcast_attrs(self, obj, names, src=0):
        """Copy the listed attributes of `obj` from rank `src` to every rank (those it has)."""
        if self.size == 1:
            return
        box = [None]
        if self.rank == src:
            box[0] = {n: getattr(obj, n) for n in names if hasattr(obj, n)}
            big = {n: v for n, v in box[0].items() if isinstance(v, np.ndarray) and v.size > (1 << 16)}
            box[0] = {n: ((v.shape, v.dtype.str) if n in big else v) for n, v in box[0].items()}
            box.append(sorted(big))
        else:
            box.append(None)
        self.td.broadcast_object_list(box, src)
        for n, v in box[0].items():
            if n in box[1]:                      # large arrays travel as tensors, not pickles
                a = getattr(obj, n) if self.rank == src else np.empty(v[0], dtype=np.dtype(v[1]))
                v = self.broadcast_array(a, src)
            if self.rank != src:
                setattr(obj, n, v)


MODEL_ATTRS = ("means_", "_covars_", "params_vec1", "init_ou_params")
INIT_ATTRS = MODEL_ATTRS + ("labels", "labels_local")


def _geometry(lv):
    """(kind, n1, n2) of a len_vec row when it describes a dense grid of exactly N_r nodes, else None."""
    n, n1, n2, kind = int(lv[0]), int(lv[3]), int(lv[4]), int(lv[8])
    if kind == 1 and n1 >= 1 and n1 == n2 and n1 * (n1 + 1) // 2 == n:
        return (1, n1, n2)
    if kind == 0 and n1 >= 1 and n2 >= 1 and n1 * n2 == n:
        return (0, n1, n2)
    return None


def make_plan(len_vec, world):
    """-> (whole[rank] = [region ids], banded = {region id: [(rank, row0, row1)] in row order}).
    Regions whose len_vec row carries the grid geometry go through `dist.plan_shards` (a region holding
    more than 1/world of the nodes is cut into row bands); without geometry regions stay whole."""
    num_region = len(len_vec)
    geo = [_geometry(lv) for lv in len_vec]
    whole = [[] for _ in range(world)]
    banded = {}
    if world > 1 and all(g is not None for g in geo):
        plan = pdist.plan_shards(geo, world)
        pieces = {}
        for rank, plist in enumerate(plan):
            for rid, r0, r1, _ in plist:
                pieces.setdefault(rid, []).append((rank, r0, r1))
        for rid, plist in pieces.items():
            if len(plist) == 1:
                whole[plist[0][0]].append(rid)
            else:
                banded[rid] = sorted(plist, key=lambda p: p[1])
    else:
        owner = pdist.assign_regions([lv[0] for lv in len_vec], world)
        for rid in range(num_region):
            whole[owner[rid]].append(rid)
    for w in whole:
        w.sort()
    return whole, banded


def band_window(kind, n1, n2, row0, row1):
    """Node ranges (region-local) of a band: owned [own0, own1) and its label window [win0, win1)
    (one halo row either side, clipped to the region)."""
    sizes = pdist.region_row_sizes(kind, n1, n2)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    h0, h1 = max(row0 - 1, 0), min(row1 + 1, len(sizes))
    return int(starts[row0]), int(starts[row1]), int(starts[h0]), int(starts[h1])


def empty_summary(n):
    """Posterior summary of n nodes that have none: map_state -1, the probabilities and entropy NaN."""
    return dict(map_state=np.full(n, -1, dtype=np.int32), map_prob=np.full(n, np.nan), label_prob=np.full(n, np.nan),
                entropy=np.full(n, np.nan))


def _gather_summary(model, len_vec, banded, label_owner, comm, n_samples):
    """The posterior summary every rank computed for its pieces, on every rank: a whole region from the rank
    that holds it, each band's owned rows from the band's rank."""
    out = empty_summary(n_samples)
    for rid in range(len(len_vec)):
        s1, s2 = int(len_vec[rid][1]), int(len_vec[rid][2])
        if rid in banded:
            kind, n1, n2 = _geometry(len_vec[rid])
            pieces = [(rank, bi) + band_window(kind, n1, n2, r0, r1)[:2] for bi, (rank, r0, r1) in enumerate(banded[rid])]
        else:
            pieces = [(label_owner[rid], None, 0, s2 - s1)]
        for rank, bi, own0, own1 in pieces:
            if rank == comm.rank:
                got = model._summary_get(rid) if bi is None else model._band_summary_get(rid, bi)
                for name, v in got.items():
                    out[name][s1 + own0:s1 + own1] = v
            for v in out.values():
                v[s1 + own0:s1 + own1] = comm.broadcast_array(np.ascontiguousarray(v[s1 + own0:s1 + own1]), rank)
    return out


def run(model, X, len_vec, threshold, annotation, m_iter, lengths=None, n_threads=None, posterior_summary=False):
    """`fit_accumulate_test` (base.py:301-455): returns (params_vec, params_vec1, params_vecList,
    iter_id1, iter_id2, cost_vec, t_labels).  posterior_summary: on every iteration that sets a new settled
    best (the one whose labels become t_labels) the summary kernel runs on each of the rank's regions and bands
    while their log-likelihood and labels are that iteration's; the pieces are gathered once, at the end, into
    ``model.posterior_summary_``."""
    comm = Comm()
    if comm.rank == 0:
        model._init(X, lengths=lengths)
    comm.broadcast_attrs(model, INIT_ATTRS)
    model._check()

    num_region = len(len_vec)
    sizes = np.array([lv[0] for lv in len_vec], dtype=np.float64)
    n_samples = int(sizes.sum())
    ratio = sizes * 1.0 / n_samples                       # base.py:332-337
    whole, banded = make_plan(len_vec, comm.size)
    mine = whole[comm.rank]
    label_owner = [None] * num_region                      # the rank that runs the region's graph cut
    for rank, ids in enumerate(whole):
        for rid in ids:
            label_owner[rid] = rank
    for rid, plist in banded.items():
        label_owner[rid] = plist[0][0]
    if banded:
        model._prepare_bands(X, len_vec, banded, comm)
    workers = n_threads or min(num_region, 8)

    K, d = model.n_components, model.n_features
    n_stat = K + K * d + K * d * d
    width = n_stat + 4 + 3                                 # statistics | 4 costs (whole) | 3 cost sums (banded)

    history = CostHistory(threshold)
    params_best = model.params_vec1.copy()
    params_settled = model.params_vec1.copy()
    params_trace = []
    t_labels = np.zeros(n_samples)
    have_summary = False

    for it in range(m_iter):
        model._sync_model()
        table = np.zeros((num_region, width))
        labels = np.zeros(n_samples)

        # ---- whole regions of this rank: the reference's per-region unit, on a thread pool
        out = _queue.Queue()
        model.queue = out
        if workers > 1 and len(mine) > 1:
            with ThreadPoolExecutor(max_workers=workers) as pool:
                list(pool.map(lambda r: model._predict_posteriors(X, len_vec, r, out), mine))
        else:
            for rid in mine:
                model._predict_posteriors(X, len_vec, rid, out)
        for _ in range(len(mine)):
            rid, stats, lab, c_raw, c_pair, c_unary, c_total = out.get()
            table[rid, :n_stat] = np.concatenate([np.ravel(stats['post']), np.ravel(stats['obs']),
                                                  np.ravel(stats['obs*obs.T'])])
            table[rid, n_stat:n_stat + 4] = (c_raw, c_pair, c_unary, c_total)
            labels[int(len_vec[rid][1]):int(len_vec[rid][2])] = lab

        # ---- regions cut into row bands: every rank takes part, one region after the other
        for rid in sorted(banded):
            part, lab = model._banded_region(rid, len_vec, banded[rid], comm)
            table[rid, :n_stat] += part[:n_stat]
            table[rid, n_stat + 4:] += part[n_stat:]
            if lab is not None:
                labels[int(len_vec[rid][1]):int(len_vec[rid][2])] = lab

        table = comm.sum(table)                            # the parent's queue sums, base.py:384-396

        stats = model._initialize_sufficient_statistics()
        raw = pairwise = unary = total = 0
        for rid in range(num_region):                      # fixed order: the sums do not depend on timing
            row = table[rid]
            costs = row[n_stat:n_stat + 4]
            if rid in banded:
                costs = costs_from_sums(row[n_stat + 4:], len_vec[rid][0])
            raw += costs[0] * ratio[rid]
            pairwise += costs[1] * ratio[rid]
            unary += costs[2] * ratio[rid]
            total += costs[3] * ratio[rid]
            stats = model._accumulate_sufficient_statistics_1(stats, {
                'post': row[:K], 'obs': row[K:K + K * d].reshape(K, d),
                'obs*obs.T': row[K + K * d:n_stat].reshape(K, d, d)})

        params_trace.append(model.params_vec1.copy())
        model.labels = labels.copy()
        is_best, is_settled, stop = history.add(it, pairwise, unary, total)
        if is_best:
            params_best = model.params_vec1.copy()
            model.labels_local = model.labels.copy()       # the next graph cuts start from here (phylo_hmrf.py:479)
        if is_settled:
            params_settled = model.params_vec1.copy()
            t_labels = model.labels.copy()
            if posterior_summary:
                for rid in mine:
                    model._summary_launch(rid)
                for rid in sorted(banded):
                    for bi, (rank, _, _) in enumerate(banded[rid]):
                        if rank == comm.rank:
                            model._band_summary_launch(rid, bi)
                have_summary = True
        if stop:
            break
        if comm.rank == 0:
            model._do_mstep(stats)
        comm.broadcast_attrs(model, MODEL_ATTRS)

    if comm.size > 1:       # every rank ends with the labels of all regions, like the reference's parent process
        for rid in range(num_region):
            s1, s2 = int(len_vec[rid][1]), int(len_vec[rid][2])
            for arr in (t_labels, model.labels, model.labels_local):
                arr[s1:s2] = comm.broadcast_array(np.ascontiguousarray(arr[s1:s2]), label_owner[rid])
    model.posterior_summary_ = None
    if posterior_summary:
        model.posterior_summary_ = (_gather_summary(model, len_vec, banded, label_owner, comm, n_samples)
                                    if have_summary else empty_summary(n_samples))
    model.params_vec1 = params_settled.copy()
    model._ou_param_varied_constraint(params_best)
    return (params_best, params_settled, np.asarray(params_trace), history.best[0], history.best_settled[0],
            np.asarray(history.rows), t_labels)
