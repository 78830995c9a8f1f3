"""Parity of the CUDA path (through the C ABI) with the CPU oracle and with the fixtures
produced by the reference's own code.  Tolerances are BASELINE.md section 5:

* FP64 log-likelihoods, statistics and cost scalars: <= 1e-9 relative;
* integer cost arrays: bit-identical except entries within 1e-9 (relative, in scaled
  units) of a truncation boundary, and those must be in the list the kernel reports;
* GCO labels: identical whenever the integer arrays are identical.
"""
import os

import numpy as np
import pytest

from oracle import phmrf_oracle as orc

pytestmark = pytest.mark.gpu

RTOL = 1e-9


@pytest.fixture(scope="module")
def ph():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import phylo_hmrf_b200 as ph
    return ph


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = np.maximum(np.abs(b), 1e-300)
    return float(np.max(np.abs(a - b) / scale)) if a.size else 0.0


def _assert_stats_close(got, ref, rtol=RTOL):
    for key in ("post", "obs", "obs*obs.T"):
        # elementwise relative, with an absolute floor tied to the array's own scale (entries
        # that are sums of cancelling-free non-negative terms can still be exactly 0)
        floor = rtol * 1e-3 * np.abs(ref[key]).max()
        np.testing.assert_allclose(got[key], ref[key], rtol=rtol, atol=floor, err_msg=key)


def _check_unary(u_gpu, logprob_gpu, logprob_ref, dwf_gpu, blist, w, V):
    # (1) the quantiser itself is bit-exact on identical inputs
    u_same, _, _, _ = orc.pygco_quantise(-logprob_gpu, w, V, down_weight_factor=dwf_gpu)
    assert np.array_equal(u_gpu, u_same)
    # (2) against the oracle's own log-likelihood only listed boundary entries may differ
    u_ref, _, _, dwf_ref = orc.pygco_quantise(-logprob_ref, w, V)
    assert abs(dwf_gpu - dwf_ref) <= 1e-12 * dwf_ref
    diff = np.flatnonzero(u_gpu.ravel() != u_ref.ravel())
    assert set(diff.tolist()) <= set(blist.tolist())
    assert np.all(np.abs(u_gpu.ravel()[diff].astype(np.int64) - u_ref.ravel()[diff]) <= 1)
    # (3) the list is what the contract says it is
    mask = orc.unary_boundary_mask(-logprob_gpu, dwf_gpu, 1e-9).ravel()
    assert set(np.flatnonzero(mask).tolist()) == set(blist.tolist())


def test_golden_fixtures_end_to_end(ph, golden):
    K, d = int(golden["K"]), int(golden["d"])
    et = int(golden["estimate_type"])
    V = golden["ref_V"]
    m = ph.Model(K, d)
    m.set_model(golden["means"], golden["covars"], V)
    for r in range(int(golden["n_regions"])):
        p = "r%d_" % r
        s1, s2 = golden["len_vec"][r][1:3]
        X = golden["X"][s1:s2]
        w, ids = golden[p + "ref_edge_w"], golden[p + "ref_edge_ids"]
        reg = m.region(X, ids, w)
        absmax = reg.emit_loglik(want_absmax=True)
        lp = reg.logprob()
        assert _rel(lp, golden[p + "logprob"]) <= RTOL
        assert absmax == np.abs(lp).max()
        q = reg.quantise(boundary_cap=lp.size)
        _check_unary(q["unary_i32"], lp, golden[p + "logprob"], q["dwf"], q["boundary_idx"], w, V)
        _, w_i, V_i, _ = orc.pygco_quantise(-lp, w, V, down_weight_factor=q["dwf"])
        assert np.array_equal(q["w_i32"], w_i) and np.array_equal(q["V_i32"], V_i)
        # phase B on the labels the reference run used
        reg.set_labels(golden[p + "labels"])
        stats, sums, post = reg.estep_stats(et, want_post=True)
        np.testing.assert_allclose(post, golden[p + "ref_post"], rtol=RTOL, atol=1e-300)
        costs = ph.costs_from_sums(sums, len(X))
        np.testing.assert_allclose(costs, golden[p + "ref_costs"], rtol=RTOL, atol=1e-12)
        ref = {"post": golden[p + "ref_stats_post"], "obs": golden[p + "ref_stats_obs"],
               "obs*obs.T": golden[p + "ref_stats_obsobsT"]}
        _assert_stats_close(stats, ref)
        np.testing.assert_allclose(reg.pairwise_potential(et), golden[p + "ref_pp"], rtol=RTOL, atol=1e-15)
        reg.close()
    m.close()


def test_dropin_class_matches_reference_queue_tuple(ph, golden):
    """phyloHMRF._predict_posteriors through the re-hosted class; the graph cut runs for
    real, so the oracle is evaluated on the labels our path produced."""
    K, d = int(golden["K"]), int(golden["d"])
    et = int(golden["estimate_type"])
    R = int(golden["n_regions"])
    len_vec = golden["len_vec"].tolist()
    els = [golden["r%d_edge_list" % r] for r in range(R)]
    X = golden["X"]
    model = ph.phyloHMRF(len(X), d, beta=float(golden["beta"]), beta1=float(golden["beta1"]), observation=X,
                         edge_list_1=els, len_vec=len_vec, n_components=K, estimate_type=et)
    model.means_, model._covars_ = golden["means"], golden["covars"]
    model.labels_local = golden["init_labels"].copy()
    assert np.array_equal(model.edge_potential, golden["ref_V"])

    class Q:
        def __init__(self):
            self.items = []

        def put(self, x):
            self.items.append(x)

    q = Q()
    tot = model._initialize_sufficient_statistics()
    for r in range(R):
        p = "r%d_" % r
        s1, s2 = len_vec[r][1:3]
        assert np.array_equal(model.edge_weightList_undirected_vec[r], golden[p + "ref_edge_w"])
        assert np.array_equal(model.edge_idList_undirected_vec[r], golden[p + "ref_edge_ids"])
        flat, off = golden[p + "ref_inc_flat"], golden[p + "ref_inc_off"]
        for i in (0, len(off) // 2, len(off) - 2):
            assert model.neighbor_edgeIdx_vec[r][i] == list(flat[off[i]:off[i + 1]])
        assert model._predict_posteriors(X, len_vec, r, q) is True
        rid, stats, labels, c_pair, c_pn, c_un, c_tot = q.items[-1]
        assert rid == r
        # label identity: oracle integer arrays -> same graph cut -> same labels
        lp_ref = golden[p + "logprob"]
        u_ref, w_ref, V_ref, _ = orc.pygco_quantise(-lp_ref, golden[p + "ref_edge_w"], golden["ref_V"])
        qd = model.last_quantise
        if np.array_equal(qd["unary_i32"], u_ref) and np.array_equal(qd["w_i32"], w_ref):
            lab_ref = ph.gco_cut_int(u_ref, golden[p + "ref_edge_ids"], w_ref, V_ref, n_iter=5000, algorithm='swap',
                                     init_labels=golden["init_labels"][s1:s2])
            assert np.array_equal(labels, lab_ref)
        ref = orc.compute_posteriors_graph(golden["ref_V"], labels, lp_ref, golden[p + "ref_edge_w"],
                                           golden[p + "ref_edge_ids"], None, et, faithful=False)
        np.testing.assert_allclose([c_pair, c_pn, c_un, c_tot], ref[1:], rtol=RTOL, atol=1e-12)
        _assert_stats_close(stats, orc.sufficient_statistics(ref[0], X[s1:s2]))
        tot = model._accumulate_sufficient_statistics_1(tot, stats)
        # the other re-hosted signatures
        post, *costs = model._compute_posteriors_graph(X[s1:s2], labels, lp_ref, r)
        np.testing.assert_allclose(post, ref[0], rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(costs, ref[1:], rtol=RTOL, atol=1e-12)
        lp = model._compute_log_likelihood(X[s1:s2])
        assert _rel(lp, lp_ref) <= RTOL
        pc = model._pairwise_compare_ensemble(labels, None, model.edge_weightList_undirected_vec[r],
                                              model.edge_idList_undirected_vec[r])
        np.testing.assert_allclose(pc, ref[1], rtol=RTOL, atol=1e-12)
        st, lpr = model.predict(X[s1:s2], r)
        assert np.array_equal(st, labels) and _rel(lpr, lp_ref) <= RTOL
    assert tot["post"].sum() == pytest.approx(len(X), rel=1e-9)
    model.close()


CASES = [
    # B, d, K, estimate_type, beta, potts
    (97, 5, 20, 3, 1.0, True),
    (97, 9, 30, 3, 1.0, True),
    (64, 4, 10, 0, 2.0, True),
    (50, 9, 40, 3, 0.5, True),     # K beyond one stat-phase pass
    (41, 1, 3, 3, 1.0, True),
    (37, 12, 7, 3, 1.0, True),
    (45, 2, 1, 3, 1.0, True),      # single state
    (60, 5, 20, 3, 1.0, False),    # general (non-Potts) compatibility matrix
    (60, 3, 6, 0, 1.0, False),
    (40, 3, 5, 3, -0.8, True),     # repulsive coupling: slot factors below 1
    (33, 9, 30, 0, 1.3, True),     # unweighted estimate on the headline shape
]


@pytest.mark.parametrize("B,d,K,et,beta,potts", CASES)
def test_random_regions_against_oracle(ph, B, d, K, et, beta, potts):
    from phylo_hmrf_b200 import synth
    seed = 1000 + B + d + K
    g = synth.make_band(seed, B, d)
    X, e, w = g["X_own"], g["edge_ids"], g["edge_w"]
    # knock out every edge of a few nodes: isolated nodes take the unweighted V row
    iso = np.array([3, len(X) // 2, len(X) - 1])
    keep = ~(np.isin(e[:, 0], iso) | np.isin(e[:, 1], iso))
    e, w = e[keep], w[keep]
    means, covars = synth.model(seed, X, K, d)
    rng = np.random.default_rng(seed)
    if potts:
        V = synth.potts(K, beta)
    else:
        A = rng.random((K, K))
        V = beta * (A + A.T)
        np.fill_diagonal(V, 0.0)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    reg = m.region(X, e, w)
    reg.emit_loglik()
    lp = reg.logprob()
    lp_ref = orc.compute_log_likelihood(X, means, covars)
    assert _rel(lp, lp_ref) <= RTOL
    q = reg.quantise(boundary_cap=lp.size)
    _check_unary(q["unary_i32"], lp, lp_ref, q["dwf"], q["boundary_idx"], w, V)
    lab = reg.labels_argmin_unary()
    assert np.array_equal(lab, np.argmin(q["unary_i32"], axis=1))
    lab = lab.copy()
    flips = rng.random(len(lab)) < 0.1
    lab[flips] = rng.integers(0, K, size=int(flips.sum()))
    reg.set_labels(lab)
    stats, sums, post = reg.estep_stats(et, want_post=True)
    ref = orc.compute_posteriors_graph(V, lab, lp_ref, w, e, None, et, faithful=False, stable=True)
    np.testing.assert_allclose(post, ref[0], rtol=RTOL, atol=1e-290)
    np.testing.assert_allclose(ph.costs_from_sums(sums, len(X)), ref[1:], rtol=RTOL, atol=1e-12)
    _assert_stats_close(stats, orc.sufficient_statistics(ref[0], X))
    np.testing.assert_allclose(reg.pairwise_potential(et), orc.pairwise_compare_vec(V, lab, w, e, et), rtol=RTOL,
                               atol=1e-15)
    # determinism: fixed-order reductions give bit-identical repeats
    stats2, sums2, _ = reg.estep_stats(et)
    for k in stats:
        assert np.array_equal(stats[k], stats2[k])
    assert np.array_equal(sums, sums2)
    reg.close()
    m.close()


def test_row_bands_add_up_to_the_whole_region(ph):
    """Sharding by contact-map row band: shared dwf (max over bands), halo labels, and the
    per-band statistics / cost sums add up to the single-region result."""
    from phylo_hmrf_b200 import synth
    B, d, K, et, seed = 120, 5, 12, 3, 77
    whole = synth.make_band(seed, B, d)
    means, covars = synth.model(seed, whole["X_own"], K, d)
    V = synth.potts(K, 1.0)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    reg = m.region(whole["X_own"], whole["edge_ids"], whole["edge_w"])
    reg.emit_loglik()
    q = reg.quantise()
    lab = reg.labels_argmin_unary()
    stats, sums, _ = reg.estep_stats(et)
    bands, absmax = [], []
    for r0, r1 in synth.band_rows(B, 3):
        g = synth.make_band(seed, B, d, r0, r1)
        b = m.region(g["X_own"], g["edge_ids"], g["edge_w"], n_window=g["n_window"], own_offset=g["own_offset"])
        absmax.append(b.emit_loglik(want_absmax=True))
        bands.append((g, b))
    wmax = max(np.abs(g["edge_w"]).max() for g, _ in bands)
    dwf = max(max(absmax), wmax * V.max()) + 1e-10
    assert dwf == q["dwf"]
    tot = None
    tot_sums = np.zeros(3)
    for g, b in bands:
        qb = b.quantise(dwf=dwf)
        o0 = g["win_start"] + g["own_offset"]
        assert np.array_equal(qb["unary_i32"], q["unary_i32"][o0:o0 + g["n_own"]])
        b.set_labels(lab[g["win_start"]:g["win_start"] + g["n_window"]])
        st, su, _ = b.estep_stats(et)
        tot = st if tot is None else {k: tot[k] + st[k] for k in st}
        tot_sums += su
        b.close()
    _assert_stats_close(tot, stats, rtol=1e-12)
    np.testing.assert_allclose(tot_sums, sums, rtol=1e-12)
    reg.close()
    m.close()


def test_edge_cases(ph):
    # one node, no edges; n not a multiple of the warp; K=2, d=2
    m = ph.Model(2, 2)
    means = np.array([[0.0, 0.0], [1.0, 1.0]])
    covars = np.stack([np.eye(2), np.array([[2.0, 0.3], [0.3, 1.0]])])
    V = np.array([[0.0, 1.5], [1.5, 0.0]])
    m.set_model(means, covars, V)
    for n in (1, 31, 33, 65):
        rng = np.random.default_rng(n)
        X = rng.random((n, 2))
        e = np.array([[i, i + 1] for i in range(n - 1)], dtype=np.int64).reshape(-1, 2)
        w = rng.random(len(e))
        reg = m.region(X, e, w)
        reg.emit_loglik()
        lp_ref = orc.compute_log_likelihood(X, means, covars)
        assert _rel(reg.logprob(), lp_ref) <= RTOL
        lab = rng.integers(0, 2, size=n)
        reg.set_labels(lab)
        stats, sums, post = reg.estep_stats(3, want_post=True)
        ref = orc.compute_posteriors_graph(V, lab, lp_ref, w, e, None, 3, faithful=False, stable=True)
        np.testing.assert_allclose(post, ref[0], rtol=RTOL)
        np.testing.assert_allclose(ph.costs_from_sums(sums, n), ref[1:], rtol=RTOL, atol=1e-12)
        _assert_stats_close(stats, orc.sufficient_statistics(ref[0], X))
        with pytest.raises(ValueError):
            reg.set_labels(np.full(n, 2))
        reg.close()
    # covariance validation mirrors the reference's ValueError
    with pytest.raises(ValueError):
        m.set_model(means, np.stack([np.eye(2), np.array([[1.0, 2.0], [2.0, 1.0]])]), V)
    # sklearn's +1e-7*I retry on a singular covariance
    sing = np.stack([np.eye(2), np.array([[1.0, 1.0], [1.0, 1.0]])])
    m.set_model(means, sing, V)
    reg = m.region(np.array([[0.2, 0.1]]), np.zeros((0, 2), np.int64), np.zeros(0))
    reg.emit_loglik()
    np.testing.assert_allclose(reg.logprob(), orc.compute_log_likelihood(np.array([[0.2, 0.1]]), means, sing),
                               rtol=1e-6)
    reg.close()
    m.close()


def test_native_library_is_the_one_loaded(ph):
    """The extension in-tree is what the process mapped (no silent fallback)."""
    maps = open("/proc/self/maps").read()
    assert "phylo_hmrf_b200/lib/libphmrf.so" in maps
    from phylo_hmrf_b200 import engine
    assert engine.launch_count() > 0


def test_quantiser_division_is_correctly_rounded(ph):
    """The integer unary must equal numpy's ((u / dwf) * 1e5).astype(intc) bit for bit on
    identical inputs: exercise the refinement-based division with adversarial magnitudes and
    many different down-weight factors (injected log-likelihoods, dwf override)."""
    rng = np.random.default_rng(123)
    K, d, n = 16, 2, 4096
    m = ph.Model(K, d)
    m.set_model(np.zeros((K, d)), np.stack([np.eye(d)] * K), np.zeros((K, K)))
    reg = m.region(np.zeros((n, d)), np.zeros((0, 2), np.int64), np.zeros(0))
    for trial in range(12):
        mag = 10.0 ** rng.uniform(-3, 6, size=(n, K))
        lp = -mag * rng.uniform(0.5, 1.0, size=(n, K)) * np.where(rng.random((n, K)) < 0.1, -1.0, 1.0)
        if trial % 3 == 0:  # values sitting on / next to truncation boundaries
            dwf = float(np.abs(lp).max() * rng.uniform(1.0, 1.5))
            ints = rng.integers(-99999, 99999, size=(n, K))
            lp = -(ints / 1e5) * dwf
            lp = np.nextafter(lp, np.where(rng.random((n, K)) < 0.5, np.inf, -np.inf))
        else:
            dwf = float(np.abs(lp).max() * rng.uniform(1.0, 3.0) + 1e-10)
        reg.set_logprob(lp)
        q = reg.quantise(dwf=dwf, want_edges=False, boundary_cap=n * K)
        ref = ((-lp / dwf) * 100000).astype(np.intc)
        assert q["dwf"] == dwf
        assert np.array_equal(q["unary_i32"], ref)
        mask = orc.unary_boundary_mask(-lp, dwf, 1e-9).ravel()
        assert set(np.flatnonzero(mask).tolist()) == set(q["boundary_idx"].tolist())
    reg.close()
    m.close()
