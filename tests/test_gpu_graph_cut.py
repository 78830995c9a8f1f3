"""The alpha-beta swap on the device (kernels_cut.cu: phmrf_graph_cut_swap, phmrf_region_graph_cut) gives the
labels and energies of the host cut (csrc/gco.cpp) on the same integer arrays: every move takes the smallest
sink side of all minimum cuts, which depends on the energy alone."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def ph():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import phylo_hmrf_b200 as ph
    return ph


def _both(ph, u, e, w, V, n_iter, init):
    lab_h, en_h, en0_h = ph.gco_cut_int(u, e, w, V, n_iter=n_iter, algorithm='swap', init_labels=init,
                                        return_energy=True)
    lab_d, en_d, en0_d = ph.gco_swap_device(u, e, w, V, n_iter=n_iter, init_labels=init, return_energy=True)
    np.testing.assert_array_equal(lab_d, lab_h)
    assert (en_d, en0_d) == (en_h, en0_h)
    return lab_h, en_h


def _problem(rng, n, K, kind, p_edge=0.35):
    """The generator of test_gco.py::test_labels_follow_the_move_rule_on_ties, with three kinds of V."""
    e = np.asarray([(i, j) for i in range(n) for j in range(i + 1, n) if rng.random() < p_edge],
                   dtype=np.int64).reshape(-1, 2)
    w = rng.integers(0, 6, len(e)).astype(np.int32)
    unary = rng.integers(0, 8, (n, K)).astype(np.int32)
    if kind == "symmetric":
        M = rng.integers(0, 4, (K, K))
        V = (M + M.T) * (1 - np.eye(K, dtype=np.int64))
    elif kind == "asymmetric":      # V[a][b] + V[b][a] >= V[a][a] + V[b][b], V[a][b] != V[b][a]
        V = rng.integers(0, 4, (K, K)) * (1 - np.eye(K, dtype=np.int64))
    else:
        V = int(rng.integers(1, 3)) * (1 - np.eye(K, dtype=np.int64))
    return unary, e, w, V.astype(np.int32)


def test_tie_heavy_problems_match_the_host_cut(ph):
    rng = np.random.default_rng(20261020)
    count = 0
    for t in range(330):
        kind = ("symmetric", "asymmetric", "potts")[t % 3]
        n_iter = (0, 1, 2, 50, -1)[t % 5]
        n, K = int(rng.integers(2, 14)), int(rng.integers(2, 6))
        u, e, w, V = _problem(rng, n, K, kind)
        init = (None, rng.integers(0, K, n).astype(np.int32), np.argmin(u, axis=1).astype(np.int32))[(t // 3) % 3]
        _both(ph, u, e, w, V, n_iter, init)
        count += 1
    # K = 1, an isolated site, degree far above 8, K = 40, no edges at all
    u, e, w, V = _problem(rng, 9, 1, "potts")
    _both(ph, u, e, w, V, -1, None)
    u, e, w, V = _problem(rng, 30, 3, "asymmetric", p_edge=0.0)
    e = np.asarray([(0, j) for j in range(1, 25)] + [(3, 7), (7, 9)], dtype=np.int64)   # sites 25..29 isolated
    w = rng.integers(0, 6, len(e)).astype(np.int32)
    _both(ph, u, e, w, V, 50, rng.integers(0, 3, 30).astype(np.int32))
    u, e, w, V = _problem(rng, 60, 40, "symmetric", p_edge=0.3)
    _both(ph, u, e, w, V, -1, rng.integers(0, 40, 60).astype(np.int32))
    _both(ph, u, np.zeros((0, 2), np.int64), np.zeros(0, np.int32), V, 5, None)
    assert count >= 300


@pytest.mark.parametrize("case", ["b56_k10", "b40_k20"])
def test_pinned_labels_of_quantised_regions(ph, case):
    from phylo_hmrf_b200 import synth
    G = np.load(os.path.join(HERE, "golden", "gco_regions.npz"))
    u, w, V = G[case + "_unary"], G[case + "_w"], G[case + "_V"]
    B = int(case[1:case.index("_")])
    e = synth.triangle_band(B, 0, B)["edge_ids"]
    init = np.argmin(u, axis=1).astype(np.int32)
    lab, en, _ = ph.gco_swap_device(u, e, w, V, n_iter=5000, init_labels=init, return_energy=True)
    assert en == int(G[case + "_swap5000_energy"])
    np.testing.assert_array_equal(lab, G[case + "_swap5000_labels"])


def _quantised_region(ph, B, K, d, seed, grid):
    from phylo_hmrf_b200 import synth
    g = synth.make_band(seed, B, d)
    means, covars = synth.model(seed, g["X_own"], K, d)
    m = ph.Model(K, d)
    m.set_model(means, covars, synth.potts(K, 1.0))
    if grid:
        r = m.region_grid(g["X_window"], 1, B, B, num_neighbor=8, beta1=0.1)
        r.set_edge_weights(g["edge_w"])
    else:
        r = m.region(g["X_own"], g["edge_ids"], g["edge_w"])
    r.emit_loglik()
    return m, r, g


@pytest.mark.parametrize("B,grid", [(200, True), (652, True), (120, False)])
def test_region_cut_leaves_the_unary_on_the_device(ph, B, grid):
    """The region's own arrays, cut where they are: the labels of the host cut on the downloaded arrays, and the
    E-step reads them without set_labels."""
    K, d = 10, 4
    m, r, g = _quantised_region(ph, B, K, d, 7 + B, grid)
    try:
        bytes0 = r.device_bytes()
        q = r.quantise()
        init = np.argmin(q["unary_i32"], axis=1).astype(np.int32)
        lab, en, en0 = r.graph_cut(init, n_iter=5000, return_energy=True)
        assert r.device_bytes() > bytes0                     # the cut's scratch is the region's
        lab_h, en_h, en0_h = ph.gco_cut_int(q["unary_i32"], g["edge_ids"], q["w_i32"], q["V_i32"], n_iter=5000,
                                            algorithm='swap', init_labels=init, return_energy=True)
        np.testing.assert_array_equal(lab, lab_h)
        assert (en, en0) == (en_h, en0_h)
        s1, c1, _ = r.estep_stats(3)
        r.set_labels(lab)
        s2, c2, _ = r.estep_stats(3)
        for k in s1:
            np.testing.assert_array_equal(s1[k], s2[k])
        np.testing.assert_array_equal(c1, c2)
        # a second cut on the same region (scratch reused) from the all-zero start, labels not downloaded
        r.quantise(want_unary=False, want_edges=False)
        lab0, en_z, _ = r.graph_cut(None, n_iter=3, return_energy=True)
        lab_hz, en_hz, _ = ph.gco_cut_int(q["unary_i32"], g["edge_ids"], q["w_i32"], q["V_i32"], n_iter=3,
                                          algorithm='swap', return_energy=True)
        np.testing.assert_array_equal(lab0, lab_hz)
        assert en_z == en_hz
    finally:
        r.close()
        m.close()


def test_errors(ph):
    from phylo_hmrf_b200 import _lib
    rng = np.random.default_rng(3)
    u, e, w, V = _problem(rng, 8, 3, "symmetric", p_edge=0.5)
    big = u.copy()
    big[5, 1] = 20000000
    init = np.ones(8, np.int32)      # label 1 is active in the first executed moves
    for cut in (lambda **k: ph.gco_cut_int(big, e, w, V, algorithm='swap', init_labels=init, **k),
                lambda **k: ph.gco_swap_device(big, e, w, V, init_labels=init, **k)):
        with pytest.raises(RuntimeError, match="GCO.*GCO_MAX_ENERGYTERM"):
            cut(n_iter=1)
        cut(n_iter=0)
    with pytest.raises(ph.PhmrfError) as ei:
        ph.gco_swap_device(u, e, -np.ones_like(w), V)
    assert ei.value.code == _lib.PHMRF_E_UNSUPPORTED
    nonsub = np.asarray([[0, 1, 0], [1, 5, 1], [0, 1, 5]], np.int32)
    with pytest.raises(ph.PhmrfError) as ei:
        ph.gco_swap_device(u, e, w, nonsub)
    assert ei.value.code == _lib.PHMRF_E_UNSUPPORTED
    with pytest.raises(RuntimeError, match="GCO.*init label"):
        ph.gco_swap_device(u, e, w, V, init_labels=np.full(8, 3, np.int32))
    with pytest.raises(RuntimeError, match="id1 < id2"):
        ph.gco_swap_device(u, np.asarray([[2, 1]]), np.ones(1, np.int32), V)
    # a region: bad init label; a band is refused
    m, r, g = _quantised_region(ph, 30, 4, 3, 1, True)
    try:
        r.quantise(want_unary=False, want_edges=False)
        with pytest.raises(RuntimeError, match="init label"):
            r.graph_cut(np.full(r.n, 4, np.int32))
        from phylo_hmrf_b200 import synth
        band = m.region_grid(g["X_window"][:synth.tri_row_start(30, 6)], 1, 30, 30, row0=0, row1=5, num_neighbor=8,
                             beta1=0.1)
        try:
            band.emit_loglik()
            band.quantise(want_unary=False, want_edges=False)
            with pytest.raises(ph.PhmrfError) as ei:
                band.graph_cut(None)
            assert ei.value.code == _lib.PHMRF_E_INVALID
        finally:
            band.close()
    finally:
        r.close()
        m.close()


def _two_region_em(graph_cut):
    """test_gpu_em.py's two-region problem and hooks; returns what fit_accumulate_test ends with."""
    import phylo_hmrf_b200 as ph
    from phylo_hmrf_b200 import synth, utility
    d, K, seed = 4, 5, 99
    regs = [synth.make_band(seed + r, B, d) for r, B in enumerate((40, 33))]
    X = np.concatenate([g["X_own"] for g in regs])
    len_vec, els, s = [], [], 0
    for r, g in enumerate(regs):
        n = g["n_own"]
        len_vec.append([n, s, s + n, g["B"], g["B"], 0, 0, r, 1, 21 + r])
        els.append(utility.edge_weightlist_grid3_undirected_unsym(g["X_own"], g["x"] * g["B"] + g["y"], g["B"], '', 8))
        s += n
    model = ph.phyloHMRF(len(X), d, beta=1.0, beta1=0.1, observation=X, edge_list_1=els, len_vec=len_vec,
                         n_components=K, estimate_type=3, graph_cut=graph_cut)
    seen = []

    def init_fn(m, Xall):
        rng = np.random.default_rng(0)
        m.means_ = Xall[rng.choice(len(Xall), K, replace=False)].copy()
        cv = np.cov(Xall.T) + m.min_covar * np.eye(d)
        m._covars_ = np.stack([cv] * K)
        m.params_vec1 = np.zeros((K, 3))
        d2 = ((Xall[:, None, :] - m.means_[None]) ** 2).sum(-1)
        m.labels = np.argmin(d2, axis=1).astype(np.int64)
        m.labels_local = m.labels.copy()

    def mstep_fn(m, stats):
        post = np.maximum(stats['post'], 1e-8)
        mu = stats['obs'] / post[:, None]
        cv = stats['obs*obs.T'] / post[:, None, None] - mu[:, :, None] * mu[:, None, :]
        m.means_ = mu
        m._covars_ = 0.5 * (cv + cv.transpose(0, 2, 1)) + m.min_covar * np.eye(d)
        m.params_vec1 = m.params_vec1 + 1.0
        seen.append({k: v.copy() for k, v in stats.items() if isinstance(v, np.ndarray)})

    model.init_fn, model.mstep_fn = init_fn, mstep_fn
    res = model.fit_accumulate_test(X, len_vec, 1e-3, "test", 12)
    q = model.last_quantise
    model.close()
    return res, seen, q


def test_em_with_the_device_cut_equals_the_host_cut(ph):
    (_, _, _, _, _, cost_h, lab_h), seen_h, q_h = _two_region_em('host')
    (_, _, _, _, _, cost_d, lab_d), seen_d, q_d = _two_region_em('device')
    np.testing.assert_array_equal(lab_d, lab_h)
    np.testing.assert_array_equal(cost_d, cost_h)
    assert len(seen_d) == len(seen_h)
    for a, b in zip(seen_d, seen_h):
        for k in a:
            np.testing.assert_allclose(a[k], b[k], rtol=1e-12, atol=0)
    assert set(q_d) == {"dwf", "V_i32"} and "unary_i32" in q_h


def test_two_gpu_banded_region_device_cut_equals_host_cut(tmp_path):
    """A region cut into two row bands over two ranks: the owner rank runs gco_swap_device on the unary it
    assembled, and the run equals the host-cut run."""
    import socket
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    worker = os.path.join(HERE, "mgpu_cut_worker.py")
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    for mode in ("host", "device"):
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), worker, str(tmp_path), mode],
                       check=True, env=env, timeout=280)
    for rank in (0, 1):
        h = np.load(str(tmp_path / ("host_rank%d.npz" % rank)))
        d = np.load(str(tmp_path / ("device_rank%d.npz" % rank)))
        assert int(d["n_bands"]) == 1
        np.testing.assert_array_equal(d["t_labels"], h["t_labels"])
        np.testing.assert_array_equal(d["cost_vec"], h["cost_vec"])
        np.testing.assert_array_equal(d["labels_local"], h["labels_local"])
