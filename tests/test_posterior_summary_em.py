"""The EM driver's posterior summary (fit_accumulate_test(..., posterior_summary=True)) without a GPU: the
per-piece arithmetic is the NumPy reference (tests/summary_ref.py), the driver logic is the product's.
Checks that the summary belongs to the best settled iteration, that the pieces of a row-banded fit over
two and three ranks (gloo) gather to the single-process result, and that the option leaves the fit alone."""
import ctypes as C
import os
import socket
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import em_band_case as case  # noqa: E402
import summary_ref  # noqa: E402
import test_em_bands_gloo as bands  # noqa: E402

from oracle import phmrf_oracle as orc  # noqa: E402
from phylo_hmrf_b200 import engine  # noqa: E402

NAMES = ("map_state", "map_prob", "label_prob", "entropy")


class SummaryModel(bands.OracleModel):
    """The row-band test's stand-in model, plus the summary hooks of phyloHMRF computed by the reference from
    what the piece last held: the whole region's log-likelihood and labels, each band's log-likelihood and
    label window."""

    def _predict_posteriors(self, X, len_vec, rid, q):
        ids, w, V = self.edge_idList_undirected_vec[rid], self.edge_weightList_undirected_vec[rid], self.edge_potential
        s1, s2 = int(len_vec[rid][1]), int(len_vec[rid][2])
        lp = orc.compute_log_likelihood(X[s1:s2], self.means_, self._covars_)
        u, wi, Vi, _ = orc.pygco_quantise(-lp, w, V)
        labels = engine.gco_cut_int(u, ids, wi, Vi, n_iter=5000, algorithm='swap',
                                    init_labels=self.labels_local[s1:s2].astype(np.int32))
        ref = orc.compute_posteriors_graph(V, labels, lp, w, ids, None, case.ET, faithful=False, stable=True)
        self._held = getattr(self, "_held", {})
        self._held[rid] = (lp, labels)
        q.put((rid, orc.sufficient_statistics(ref[0], X[s1:s2]), labels) + tuple(ref[1:]))
        return True

    def _band_estep(self, rid, bi, labels_window):
        self._g[(rid, bi)]["labels_window"] = np.array(labels_window)
        return super()._band_estep(rid, bi, labels_window)

    def _summary_launch(self, rid):
        lp, labels = self._held[rid]
        self._sums = getattr(self, "_sums", {})
        self._sums[rid] = summary_ref.summary(self.edge_potential, labels, lp, self.edge_weightList_undirected_vec[rid],
                                              self.edge_idList_undirected_vec[rid], case.ET)

    def _summary_get(self, rid):
        return self._sums[rid]

    def _band_summary_launch(self, rid, bi):
        g = self._g[(rid, bi)]
        g["summary"] = summary_ref.summary(self.edge_potential, g["labels_window"], g["lp"], g["edge_w"],
                                           g["edge_ids"], case.ET, g["own_offset"])

    def _band_summary_get(self, rid, bi):
        return self._g[(rid, bi)]["summary"]


def _run(two_regions=False, posterior_summary=True, m_iter=bands.M_ITER):
    X, len_vec, edge_list_vec = bands._problem(two_regions)
    m = object.__new__(SummaryModel)
    m.setup(X, len_vec, edge_list_vec)
    m._region_seeds = [case.SEED, case.SEED + 1]
    m._region_bins = [bands.B, bands.B_SMALL]
    trace = []                                   # the model each iteration's E-step ran with

    def init_fn(mm, XX):
        case.init_fn(mm, XX)
        trace.append(mm.means_.copy())

    def mstep_fn(mm, stats):
        case.mstep_fn(mm, stats)
        trace.append(mm.means_.copy())

    m.init_fn, m.mstep_fn = init_fn, mstep_fn
    res = m.fit_accumulate_test(X, len_vec, 1e-12, "test", m_iter, n_threads=1, posterior_summary=posterior_summary)
    return m, res, trace, (X, len_vec, edge_list_vec)


def _worker(rank, world, port, out_dir, two_regions):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        m, res, _, _ = _run(two_regions)
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), t_labels=res[6], cost_vec=res[5],
                 **m.posterior_summary_)
    finally:
        dist.destroy_process_group()


def _assert_same_summary(a, b):
    np.testing.assert_array_equal(a["map_state"], b["map_state"])
    for k in NAMES[1:]:
        np.testing.assert_allclose(a[k], b[k], rtol=1e-12, atol=1e-15)


def test_summary_is_the_best_settled_iteration_and_leaves_the_fit_unchanged():
    m, res, trace, (X, len_vec, el) = _run(True)
    _, res_off, _, _ = _run(True, posterior_summary=False)
    for a, b in zip(res, res_off):
        np.testing.assert_array_equal(np.asarray(a), np.asarray(b))
    it = res[4]
    assert it >= 3 and len(trace) > it
    got = m.posterior_summary_
    assert set(got) == set(NAMES) and all(len(got[k]) == len(X) for k in NAMES)
    assert got["map_state"].dtype == np.int32
    t_labels = np.asarray(res[6], dtype=np.int64)
    for rid, lv in enumerate(len_vec):
        s1, s2 = int(lv[1]), int(lv[2])
        ids = np.int64(el[rid][:, :2])
        w = np.exp(-case.BETA1 * el[rid][:, 2])
        lp = orc.compute_log_likelihood(X[s1:s2], trace[it], m._covars_)
        ref = summary_ref.summary(m.edge_potential, t_labels[s1:s2], lp, w, ids, case.ET)
        summary_ref.assert_summary_close({k: v[s1:s2] for k, v in got.items()}, ref)
    # the posterior of the reported label never exceeds the MAP state's, and both lie in (0, 1]
    assert np.all(got["label_prob"] <= got["map_prob"] * (1 + 1e-12))
    assert np.all((got["map_prob"] > 0) & (got["map_prob"] <= 1 + 1e-12))
    assert np.all(got["entropy"] >= -1e-12) and np.all(got["entropy"] <= np.log(bands.K) + 1e-12)


def test_fit_without_a_settled_iteration_holds_no_summary():
    m, res, _, (X, _, _) = _run(False, m_iter=3)      # iterations 0-2 never settle
    got = m.posterior_summary_
    assert np.all(got["map_state"] == -1)
    for k in NAMES[1:]:
        assert np.all(np.isnan(got[k]))
    m2, _, _, _ = _run(False, posterior_summary=False, m_iter=3)
    assert m2.posterior_summary_ is None


@pytest.mark.parametrize("world,two_regions", [(2, False), (3, True)])
def test_gathered_summary_of_a_banded_fit_matches_the_single_process_one(tmp_path, world, two_regions):
    m1, res1, _, _ = _run(two_regions)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(world, port, str(tmp_path), two_regions), nprocs=world, join=True)
    for rank in range(world):
        got = np.load(str(tmp_path / ("rank%d.npz" % rank)))
        np.testing.assert_array_equal(got["t_labels"], res1[6])
        np.testing.assert_allclose(got["cost_vec"], res1[5], rtol=1e-10)
        _assert_same_summary(got, m1.posterior_summary_)


def test_entry_points_reject_bad_arguments_without_a_device():
    from phylo_hmrf_b200 import _lib, build
    build.build_all()
    L = _lib.lib()
    assert L.phmrf_posterior_summary(None, 0) == _lib.PHMRF_E_INVALID
    assert b"phmrf_posterior_summary" in L.phmrf_last_error()
    assert L.phmrf_get_posterior_summary(None, None, None, None, None) == _lib.PHMRF_E_INVALID
    out = np.empty(4)
    assert L.phmrf_get_posterior_summary(None, None, out.ctypes.data_as(C.POINTER(C.c_double)), None, None) == -1


def test_cli_rejects_an_unknown_summary_switch(monkeypatch):
    from phylo_hmrf_b200 import cli
    monkeypatch.setenv("PHMRF_POSTERIOR_SUMMARY", "yes")
    with pytest.raises(SystemExit, match="PHMRF_POSTERIOR_SUMMARY"):
        cli.run(cli.parse_args([]))
