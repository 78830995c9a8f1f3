"""The per-node posterior summary on the GPU (phmrf_posterior_summary) against the NumPy reference of
tests/summary_ref.py: explicit and grid-built regions and bands, any K and d, Potts and general V, both
estimate types, isolated nodes, log-likelihoods far below zero; and at fit level, the summary
fit_accumulate_test(..., posterior_summary=True) keeps for the best settled iteration."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import summary_ref  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ph():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import phylo_hmrf_b200 as ph
    return ph


def _model(ph, K, d, V, seed=0):
    rng = np.random.default_rng(seed)
    m = ph.Model(K, d)
    m.set_model(rng.normal(size=(K, d)), np.stack([np.eye(d)] * K), V)
    return m


def _V(K, potts, seed=0):
    from phylo_hmrf_b200 import synth
    if potts:
        return synth.potts(K, 0.8)
    rng = np.random.default_rng(seed)
    V = rng.uniform(0.0, 2.0, size=(K, K))
    return V + V.T


def _logp(rng, n, K, level):
    """[n,K] log-likelihoods around `level` (spread of a few hundred: many posteriors underflow)."""
    return level - rng.exponential(50.0, size=(n, K))


def _away_labels(rng, lp, K):
    """labels that are not the arg-max of the log-likelihood where K > 1."""
    am = np.argmax(lp, axis=1)
    return ((am + 1 + rng.integers(0, max(K - 1, 1), size=len(lp))) % K).astype(np.int32) if K > 1 else am.astype(np.int32)


def _check(reg, V, lab_window, lp, w, e, et, own_offset=0):
    reg.set_logprob(lp)
    reg.set_labels(lab_window)
    reg.posterior_summary(et)
    got = reg.get_posterior_summary()
    ref = summary_ref.summary(V, lab_window, lp, w, e, et, own_offset)
    # logp - pp rounds to the ulp of logp: near -2e6 that is 4.7e-10, and a last-bit difference between the two
    # sums of pp moves a_k - m, the posteriors (relative) and the entropy (absolute) by that much
    cond = 8 * np.finfo(np.float64).eps * float(np.abs(lp).max())
    summary_ref.assert_summary_close(got, ref, rtol=max(1e-9, cond), atol_entropy=max(1e-12, cond))
    return got


def _explicit_graph(rng, g, extra=0, isolated=0):
    """Window edges of a triangle band, optionally with `extra` random long-range edges (degree > 8) and
    `isolated` owned nodes cut from every edge."""
    e, w = g["edge_ids"], g["edge_w"]
    o0, n = g["own_offset"], g["n_own"]
    if extra:
        a = rng.integers(o0, o0 + n, size=extra)
        b = rng.integers(0, g["n_window"], size=extra)
        new = np.stack([np.minimum(a, b), np.maximum(a, b)], axis=1)
        new = new[new[:, 0] != new[:, 1]]
        have = set(map(tuple, e.tolist()))
        new = np.array(sorted({tuple(p) for p in new.tolist()} - have), dtype=np.int64).reshape(-1, 2)
        e = np.concatenate([e, new])
        w = np.concatenate([w, rng.uniform(0.1, 1.0, size=len(new))])
    if isolated:
        iso = rng.choice(np.arange(o0, o0 + n), size=isolated, replace=False)
        keep = ~(np.isin(e[:, 0], iso) | np.isin(e[:, 1], iso))
        e, w = e[keep], w[keep]
    return e, w


@pytest.mark.parametrize("d,K", [(1, 1), (4, 7), (9, 30), (12, 45), (4, 8), (9, 41)])
@pytest.mark.parametrize("potts", [True, False])
@pytest.mark.parametrize("et", [0, 3])
def test_explicit_region_and_band(ph, d, K, potts, et):
    from phylo_hmrf_b200 import synth
    rng = np.random.default_rng(d * 100 + K)
    V = _V(K, potts, K)
    m = _model(ph, K, d, V)
    B = 30
    for r0, r1, extra, iso in [(0, B, 0, 5), (0, B, 400, 3), (9, 17, 60, 2)]:
        g = synth.make_band(11 + K, B, d, r0, r1)
        e, w = _explicit_graph(rng, g, extra, iso)
        o0, n = g["own_offset"], g["n_own"]
        reg = m.region(g["X_own"], e, w, n_window=g["n_window"], own_offset=o0)
        for level in (-30.0, -1e6, -2e6):
            lp = _logp(rng, n, K, level)
            lab = rng.integers(0, K, size=g["n_window"]).astype(np.int32)
            lab[o0:o0 + n] = _away_labels(rng, lp, K)
            _check(reg, V, lab, lp, w, e, et, o0)
        reg.close()
    m.close()


@pytest.mark.parametrize("nn", [8, 4])
@pytest.mark.parametrize("K,et,potts", [(30, 3, True), (7, 0, False), (1, 3, True), (45, 3, False)])
def test_grid_triangle_whole_and_bands(ph, nn, K, et, potts):
    from phylo_hmrf_b200 import synth
    B, d, beta1 = 41, 9, 0.3
    rng = np.random.default_rng(K + nn)
    V = _V(K, potts, 3)
    m = _model(ph, K, d, V)
    for r0, r1 in [(0, B)] + synth.band_rows(B, 3):
        g = synth.make_band(5, B, d, r0, r1, beta1=beta1)
        rg = m.region_grid(g["X_window"], 1, B, B, r0, r1, nn, beta1)
        e, w = rg.edges()        # the device-built weights the implicit grid reads
        o0, n = rg.own_offset, rg.n
        for level in (-40.0, -1e6):
            lp = _logp(rng, n, K, level)
            lab = rng.integers(0, K, size=rg.n_window).astype(np.int32)
            lab[o0:o0 + n] = _away_labels(rng, lp, K)
            _check(rg, V, lab, lp, w, e, et, o0)
        rg.close()
    m.close()


@pytest.mark.parametrize("et,potts", [(3, True), (0, False)])
def test_grid_rectangle_whole_and_band(ph, et, potts):
    n1, n2, d, K, beta1 = 23, 31, 4, 9, 0.5
    rng = np.random.default_rng(1)
    X = np.log1p(rng.gamma(2.0, 0.5, size=(n1 * n2, d)))
    V = _V(K, potts, 4)
    m = _model(ph, K, d, V)
    r0, r1 = 5, 14
    for X_w, rows in ((X, (0, n1)), (X[(r0 - 1) * n2:(r1 + 1) * n2], (r0, r1))):
        rg = m.region_grid(X_w, 0, n1, n2, rows[0], rows[1], 8, beta1)
        e, w = rg.edges()
        o0, n = rg.own_offset, rg.n
        lp = _logp(rng, n, K, -2e6)
        lab = rng.integers(0, K, size=rg.n_window).astype(np.int32)
        lab[o0:o0 + n] = _away_labels(rng, lp, K)
        _check(rg, V, lab, lp, w, e, et, o0)
        rg.close()
    m.close()


def test_repeatable_and_leaves_the_estep_alone(ph):
    """Repeated summaries are bit-identical; running one changes neither the E-step's statistics nor those of
    the next iteration; the buffer is counted in the region's device bytes."""
    from phylo_hmrf_b200 import synth
    B, d, K, et = 40, 9, 30, 3
    g = synth.make_band(8, B, d)
    means, covars = synth.model(8, g["X_own"], K, d)
    V = synth.potts(K, 1.0)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    regs = [m.region_grid(g["X_window"], 1, B, B), m.region_grid(g["X_window"], 1, B, B)]
    lab = np.random.default_rng(0).integers(0, K, size=regs[0].n_window).astype(np.int32)
    out = []
    for with_summary, reg in zip((True, False), regs):
        reg.emit_loglik()
        reg.set_labels(lab)
        before = reg.device_bytes()
        stats = [reg.estep_stats(et)]
        if with_summary:
            reg.posterior_summary(et)
            s1 = reg.get_posterior_summary()
            assert reg.device_bytes() - before >= 28 * reg.n
            reg.posterior_summary(et)
            s2 = reg.get_posterior_summary()
            for k in s1:
                assert np.array_equal(s1[k], s2[k]) and s1[k].tobytes() == s2[k].tobytes()
        stats.append(reg.estep_stats(et))
        m.set_model(means * 1.01, covars, V)          # the next iteration
        reg.emit_loglik()
        stats.append(reg.estep_stats(et))
        m.set_model(means, covars, V)
        out.append(stats)
    for (sa, ua, _), (sb, ub, _) in zip(*out):
        assert ua.tobytes() == ub.tobytes()
        assert all(sa[k].tobytes() == sb[k].tobytes() for k in sa)
    for reg in regs:
        reg.close()
    m.close()


def test_state_errors(ph):
    from phylo_hmrf_b200 import synth
    g = synth.make_band(3, 12, 3)
    m = _model(ph, 4, 3, synth.potts(4, 1.0))
    reg = m.region(g["X_own"], g["edge_ids"], g["edge_w"])
    with pytest.raises(ph.PhmrfError) as ei:
        reg.posterior_summary(0)                      # no log-likelihood, no labels
    assert ei.value.code == -4
    with pytest.raises(ph.PhmrfError) as ei:
        reg.get_posterior_summary()                   # nothing computed yet
    assert ei.value.code == -4
    reg.emit_loglik()
    with pytest.raises(ph.PhmrfError):
        reg.posterior_summary(0)                      # labels missing
    reg.close()
    m.close()


def _fit(ph, K, d, posterior_summary):
    from phylo_hmrf_b200 import synth, utility
    regs = [synth.make_band(61 + r, B, d) for r, B in enumerate((34, 21))]
    X = np.concatenate([g["X_own"] for g in regs])
    len_vec, els, s = [], [], 0
    for r, g in enumerate(regs):
        n = g["n_own"]
        len_vec.append([n, s, s + n, g["B"], g["B"], 0, 0, r, 1, 21 + r])
        els.append(utility.edge_weightlist_grid3_undirected_unsym(g["X_own"], g["x"] * g["B"] + g["y"], g["B"], '', 8))
        s += n
    els[1] = els[1][:-1]           # no longer the grid's edge list: the second region takes explicit slots
    model = ph.phyloHMRF(len(X), d, beta=1.0, beta1=0.1, observation=X, edge_list_1=els, len_vec=len_vec,
                         n_components=K, estimate_type=3)
    assert [type(r).__name__ for r in model._regions] == ["GridRegion", "Region"]
    trace = []

    def init_fn(m, Xall):
        m.means_, m._covars_ = synth.model(5, Xall, K, d)
        m.params_vec1 = np.zeros((K, 3))
        m.labels = np.argmin(((Xall[:, None, :] - m.means_[None]) ** 2).sum(-1), axis=1).astype(np.int64)
        m.labels_local = m.labels.copy()
        trace.append((m.means_.copy(), m._covars_.copy()))

    def mstep_fn(m, stats):
        post = np.maximum(stats['post'], 1e-8)
        mu = stats['obs'] / post[:, None]
        cv = stats['obs*obs.T'] / post[:, None, None] - mu[:, :, None] * mu[:, None, :]
        m.means_ = mu
        m._covars_ = 0.5 * (cv + cv.transpose(0, 2, 1)) + m.min_covar * np.eye(d)
        m.params_vec1 = m.params_vec1 + 1.0
        trace.append((m.means_.copy(), m._covars_.copy()))

    model.init_fn, model.mstep_fn = init_fn, mstep_fn
    res = model.fit_accumulate_test(X, len_vec, 1e-6, "test", 10, posterior_summary=posterior_summary)
    out = (res, getattr(model, "posterior_summary_", None), trace, X, len_vec, els, model.edge_potential)
    model.close()
    return out


def test_fit_keeps_the_summary_of_the_best_settled_iteration(ph):
    from oracle import phmrf_oracle as orc
    K, d = 6, 4
    res, got, trace, X, len_vec, els, V = _fit(ph, K, d, True)
    res_off, none, _, _, _, _, _ = _fit(ph, K, d, False)
    assert none is None
    for a, b in zip(res, res_off):
        assert np.asarray(a).tobytes() == np.asarray(b).tobytes()
    it = res[4]
    assert it >= 3
    means, covars = trace[it]
    t_labels = np.asarray(res[6], dtype=np.int64)
    for rid, lv in enumerate(len_vec):
        s1, s2 = int(lv[1]), int(lv[2])
        lp = orc.compute_log_likelihood(X[s1:s2], means, covars)
        ref = summary_ref.summary(V, t_labels[s1:s2], lp, np.exp(-0.1 * els[rid][:, 2]), np.int64(els[rid][:, :2]), 3)
        summary_ref.assert_summary_close({k: v[s1:s2] for k, v in got.items()}, ref, rtol=1e-8, atol_entropy=1e-9)


def test_two_gpu_banded_summary_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    worker = os.path.join(HERE, "mgpu_summary_worker.py")
    args = [str(tmp_path), "96", "5", "8", "8"]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    subprocess.run([sys.executable, worker] + args, check=True, env=env, timeout=600)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                    "--master-addr", "127.0.0.1", "--master-port", str(port), worker] + args, check=True, env=env,
                   timeout=900)
    one = np.load(str(tmp_path / "w1_rank0.npz"))
    assert np.all(one["map_state"] >= 0)
    for rank in (0, 1):
        two = np.load(str(tmp_path / ("w2_rank%d.npz" % rank)))
        assert int(two["n_bands"]) == 1
        np.testing.assert_array_equal(two["t_labels"], one["t_labels"])
        np.testing.assert_array_equal(two["map_state"], one["map_state"])
        for k in ("map_prob", "label_prob", "entropy"):
            np.testing.assert_allclose(two[k], one[k], rtol=1e-9, atol=1e-12)
