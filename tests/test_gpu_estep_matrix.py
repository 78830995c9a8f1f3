"""Phase B against the oracle across its kernel matrix.

* a Python mirror of the launch chain (BulkCfg, bulk_smem_bytes, bulk_producers, bulk_acc_fits, bulk_smem_fits,
  estep_bulk_supported in estep_bulk.cuh / kernels_b3.cu, make_plan in kernels_b.cu), pinned to the built library
  through what a caller can observe: launches of a warm E-step (the general kernel launches once per pass), the
  device bytes an explicit region adds at its first pipeline E-step (the per-slot factors, 8*W*ld), and the factor
  kernel the first E-step launches on the pipeline path only;
* every estep_bulk_kernel<D, NK8, P, GRID, KR> the library holds, on explicit-slot and grid-built regions;
* the routing limits (K, accumulator tiles, degree, coupling), each just inside and just outside;
* regions large enough that every producer warp runs three or more tiles and the last round is ragged, for P = 12
  (small and large accumulator tile), 8 and 4, on whole regions, row bands and both grid geometries;
* the general kernel with three or more passes, a non-Potts V, the pairwise potential and warps that stride;
* log-likelihoods far below zero (near and beyond the padding state's value) for odd and even K.
"""
import numpy as np
import pytest

from oracle import phmrf_oracle as orc

pytestmark = pytest.mark.gpu
RTOL = 1e-9

# ---------------------------------------------------------------------------------------------------------------
# Mirror of the library's kernel choice and launch shapes
# ---------------------------------------------------------------------------------------------------------------
K_CONS, Y_SLOTS, SMEM_MAX, EXP_TAB, FAST_SLOTS, TILE = 4, 2, 227 * 1024, 2048, 8, 32


def n_features(D):
    return 1 + D + D * (D + 1) // 2


def bulk_nt(D):
    return (n_features(D) + 7) // 8


def bulk_smem_bytes(D, NK8, P):
    return (P * (8 * NK8 * 256) + K_CONS * Y_SLOTS * (8 * bulk_nt(D) * 256) + EXP_TAB * 8
            + (3 * P + K_CONS * Y_SLOTS) * 8 + P * 3 * 8 + 256)


def bulk_producers(D, NK8):
    return 12 if bulk_smem_bytes(D, NK8, 12) <= SMEM_MAX else (8 if bulk_smem_bytes(D, NK8, 8) <= SMEM_MAX else 4)


def bulk_acc_fits(D, NK8):
    return NK8 * bulk_nt(D) * 2 <= 64


def bulk_smem_fits(D, NK8):
    return bulk_smem_bytes(D, NK8, bulk_producers(D, NK8)) <= SMEM_MAX


def nk8(K):
    return (K + 7) // 8


def bulk_kr(K):
    return min((K - 8 * (nk8(K) - 1) + 1) & ~1, 8)


def bulk_small_acc(D, K):
    """RegBudget's SMALL: the consumer holds at most 12 accumulator tiles."""
    return nk8(K) * bulk_nt(D) <= 12


def bulk_supported(D, K, W, s_bound, potts=True, pp=False):
    return (not pp and potts and 1 <= W <= FAST_SLOTS and abs(s_bound) < 100.0 and K <= 40
            and bulk_acc_fits(D, nk8(K)) and bulk_smem_fits(D, nk8(K)))


def bulk_instantiation(D, K, grid):
    return (D, nk8(K), bulk_producers(D, nk8(K)), bool(grid), bulk_kr(K))


def bulk_launch(D, K, n, sms):
    """-> (P, CTAs, tiles): launch_bulk_pk."""
    P = bulk_producers(D, nk8(K))
    n_tiles = -(-n // TILE)
    return P, max(1, min(-(-n_tiles // P), sms)), n_tiles


BULK_PAIRS = [(D, k) for D in range(1, 13) for k in range(1, 6) if bulk_acc_fits(D, k) and bulk_smem_fits(D, k)]
ALL_INSTANTIATIONS = {(D, k, bulk_producers(D, k), g, kr) for D, k in BULK_PAIRS for g in (False, True)
                      for kr in (2, 4, 6, 8)}

TILE_FOR = {1: (8, 3), 2: (8, 6), 3: (5, 10), 4: (6, 8), 5: (5, 11), 6: (4, 14), 7: (5, 12), 8: (4, 15), 9: (5, 11),
            10: (5, 11), 11: (4, 13), 12: (4, 13)}   # estep_common.cuh tile_for


def _even_up(v):
    return (v + 1) & ~1


def _pad_row(v):
    return _even_up(v) if (_even_up(v) // 2) % 2 == 1 else _even_up(v) + 2


def _tile_stride(T, ntiles):
    def ok(S):
        return all(4 <= ((t2 - t1) * S * 2) % 32 <= 28 for t1 in range(ntiles) for t2 in range(t1 + 1, ntiles))
    return next((S for S in range(_even_up(T), _even_up(T) + 17, 2) if ok(S)), _even_up(T))


def general_plan(D, K, n, sms):
    """make_plan: k tiles per pass, passes, warps per block, blocks."""
    tk, tf = TILE_FOR[D]
    F = n_features(D)
    nft = -(-F // tf)
    max_kt = 32 // nft
    tks, tfs = _tile_stride(tk, max_kt), _tile_stride(tf, nft)
    rsy = _pad_row(nft * tfs)
    nkt_total = -(-K // tk)
    nkt_pass = min(nkt_total, max_kt)
    rsp = _pad_row(nkt_total * tks)
    wpb = min(8, (220 * 1024) // (32 * (rsp + rsy) * 8))
    n_tiles = -(-n // TILE)
    grid = max(1, min(-(-n_tiles // wpb), sms))
    return dict(nkt_total=nkt_total, nkt_pass=nkt_pass, n_pass=-(-nkt_total // nkt_pass), wpb=wpb, grid=grid,
                n_tiles=n_tiles)


def test_mirror_counts():
    """416 pipeline kernels: 52 (D, NK8) pairs x 4 KR x 2 region kinds; P = 4 only at d = 12 with K = 9..16."""
    assert len(BULK_PAIRS) == 52 and len(ALL_INSTANTIATIONS) == 416
    assert [(D, k) for D, k in BULK_PAIRS if bulk_producers(D, k) == 4] == [(12, 2)]
    assert sorted((D, k) for D, k in BULK_PAIRS if bulk_producers(D, k) == 8) == [(8, 5), (10, 3), (11, 3), (12, 1)]
    assert general_plan(6, 45, 1000, 148)["n_pass"] == 1 and general_plan(9, 45, 1000, 148)["n_pass"] == 2


# ---------------------------------------------------------------------------------------------------------------
# Inputs and the reference
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ph():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import phylo_hmrf_b200 as ph
    return ph


@pytest.fixture(scope="module")
def sms(ph):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rect_edges(n_window, n2, rng, lo=0, hi=None):
    """8-neighbourhood of a row-major grid of n2 columns cut after n_window nodes (id1 < id2, sorted), keeping the
    edges with an end in [lo, hi); weights in (0.05, 1]."""
    hi = n_window if hi is None else hi
    i = np.arange(n_window, dtype=np.int64)
    c = i % n2
    cand = np.stack([i + 1, i + n2 - 1, i + n2, i + n2 + 1], axis=1)
    ok = np.stack([c < n2 - 1, c > 0, np.ones_like(c, bool), c < n2 - 1], axis=1) & (cand < n_window)
    a = np.broadcast_to(i[:, None], cand.shape)[ok]
    b = cand[ok]
    keep = ((a >= lo) & (a < hi)) | ((b >= lo) & (b < hi))
    e = np.stack([a[keep], b[keep]], axis=1)
    e = e[np.lexsort((e[:, 1], e[:, 0]))]
    return e, 0.05 + 0.95 * rng.random(len(e))


def _features(rng, n, d):
    return np.log1p(rng.gamma(2.0, 0.5, size=(n, d)))


def _reference(V, lab_window, lp, w, e, et, off, n):
    """Posteriors, the four cost scalars and the statistics' posteriors of the owned nodes [off, off+n) of a window:
    compute_posteriors_graph's arithmetic (vectorised pairwise terms, stable soft-max) restricted to them."""
    lab_window = np.asarray(lab_window, dtype=np.int64)
    if off == 0 and n == len(lab_window):
        ref = orc.compute_posteriors_graph(V, lab_window, lp, w, e, None, et, faithful=False, stable=True)
        return ref[0], np.array(ref[1:])
    pp = orc.pairwise_compare_vec(V, lab_window, w, e, et)[off:off + n]
    ww = np.asarray(w, dtype=np.float64) if et == 3 else np.ones(len(e))
    la, lb = lab_window[e[:, 0]], lab_window[e[:, 1]]
    per_node = np.zeros(len(lab_window))
    np.add.at(per_node, e[:, 1], V[la, lb] * ww)
    np.add.at(per_node, e[:, 0], V[lb, la] * ww)
    pc = per_node[off:off + n].sum() / n
    post = orc._stable_softmax(lp - pp)
    costs = orc.compute_cost_v1(lab_window[off:off + n], lp, orc._stable_softmax(-pp), pc)
    return post, np.array(costs)


def _compare(ph, post, sums, stats, X, ref_post, ref_costs, msg):
    n = len(X)
    np.testing.assert_allclose(post, ref_post, rtol=RTOL, atol=1e-290, err_msg=msg)
    np.testing.assert_allclose(ph.costs_from_sums(sums, n), ref_costs, rtol=RTOL, atol=1e-12, err_msg=msg)
    st = orc.sufficient_statistics(ref_post, X)
    for key in st:
        np.testing.assert_allclose(stats[key], st[key], rtol=RTOL, atol=RTOL * 1e-3 * np.abs(st[key]).max(),
                                   err_msg=msg + " " + key)


# ---------------------------------------------------------------------------------------------------------------
# What the library ran: launches and device bytes
# ---------------------------------------------------------------------------------------------------------------
def _observe(ph, reg, et, fresh_rowmax):
    """Two E-steps without posteriors on a region whose factors were never built: (launches of the first, launches
    of the second, device bytes the first added, statistics of both).  fresh_rowmax: the log-likelihood came from
    emission, so the first E-step also launches the per-node maxima."""
    lc = ph.engine.launch_count
    b0, c0 = reg.device_bytes(), lc()
    s1, u1, _ = reg.estep_stats(et)
    c1, b1 = lc(), reg.device_bytes()
    s2, u2, _ = reg.estep_stats(et)
    c2 = lc()
    assert all(np.array_equal(s1[k], s2[k]) for k in s1) and np.array_equal(u1, u2), "repeat E-step differs"
    return dict(first=c1 - c0 - (CAL["rowmax"] if fresh_rowmax else 0), warm=c2 - c1, grew=b1 - b0)


CAL = {}


def _kernel(ph, obs, reg=None, W=None):
    """-> ('bulk', 1) or ('general', passes) from an _observe result, by the calibrated launch counts."""
    extra = obs["first"] - obs["warm"]
    assert extra in (0, 1), obs
    if extra == 1:
        assert obs["warm"] == CAL["base"] + 1, obs
        if reg is not None and not isinstance(reg, ph.engine.GridRegion):
            ld = -(-max(reg.n, 1) // 64) * 64
            assert obs["grew"] == 8 * W * ld, obs
        return "bulk", 1
    if reg is not None and not isinstance(reg, ph.engine.GridRegion):
        assert obs["grew"] == 0, obs
    return "general", obs["warm"] - CAL["base"]


def _band_data(seed, B, d, K):
    from phylo_hmrf_b200 import synth
    g = synth.make_band(seed, B, d)
    means, covars = synth.model(seed, g["X_own"], K, d)
    return g["X_own"], g["edge_ids"], g["edge_w"], means, covars


@pytest.fixture(scope="module")
def calibrated(ph):
    """Launch counts of one known pipeline shape (d=5, K=11) and one known single-pass general shape (d=6, K=45), on
    an explicit and a grid-built region: what a warm E-step launches besides the phase-B kernel(s), and what the
    first E-step after emission adds (the per-node maxima)."""
    from phylo_hmrf_b200 import synth
    out = {}
    for d, K, kind in ((5, 11, "bulk"), (6, 45, "general")):
        X, e, w, means, covars = _band_data(31, 30, d, K)
        m = ph.Model(K, d)
        m.set_model(means, covars, synth.potts(K, 1.0))
        regs = [m.region(X, e, w), m.region_grid(X, 1, 30, 30)]
        for reg in regs:
            reg.emit_loglik()
            reg.set_labels(np.random.default_rng(0).integers(0, K, size=reg.n_window))
            lc = ph.engine.launch_count
            b0, c0 = reg.device_bytes(), lc()
            reg.estep_stats(3)
            c1, b1 = lc(), reg.device_bytes()
            reg.estep_stats(3)
            c2 = lc()
            out.setdefault(kind, []).append((c1 - c0, c2 - c1, b1 - b0, reg))
        W = int(np.bincount(e.ravel()).max())
        assert (kind == "bulk") == bulk_supported(d, K, W, 1.0 * W * np.abs(w).max())
        out[kind + "_keep"] = (m, regs, W)
    (gf, gw, gb, _), (gf2, gw2, _, _) = out["general"]
    (bf, bw, bb, rb), (bf2, bw2, _, _) = out["bulk"]
    # both region kinds launch the same; the general kernel ran one pass, the pipeline one kernel
    assert (gf, gw) == (gf2, gw2) and (bf, bw) == (bf2, bw2)
    assert bw == gw, "a warm pipeline E-step and a one-pass general E-step launch alike"
    assert bf - bw == gf - gw + 1, "the first pipeline E-step builds the per-slot factors"
    assert gb == 0 and bb == 8 * out["bulk_keep"][2] * (-(-rb.n // 64) * 64)
    CAL.update(rowmax=gf - gw, base=gw - 1)
    for kind in ("bulk", "general"):
        m, regs, _ = out[kind + "_keep"]
        for r in regs:
            r.close()
        m.close()
    return dict(CAL)


def test_calibration_shapes(ph, calibrated):
    assert calibrated["rowmax"] >= 0 and calibrated["base"] >= 1


# ---------------------------------------------------------------------------------------------------------------
# One case: build, observe the kernel, compare with the oracle
# ---------------------------------------------------------------------------------------------------------------
def _run_case(ph, m, reg, X_own, lab_window, e, w, V, et, lp_ref, W, expect, msg, set_lp=None):
    """expect: ('bulk', instantiation) or ('general', passes).  set_lp: upload this log-likelihood instead of
    emitting one."""
    if set_lp is None:
        reg.emit_loglik()
    else:
        reg.set_logprob(set_lp)
    reg.set_labels(lab_window)
    obs = _observe(ph, reg, et, fresh_rowmax=set_lp is None)
    kind, passes = _kernel(ph, obs, reg, W)
    if expect[0] == "bulk":
        assert kind == "bulk", (msg, obs)
    else:
        assert (kind, passes) == expect, (msg, obs)
    stats, sums, post = reg.estep_stats(et, want_post=True)
    off = reg.own_offset
    ref_post, ref_costs = _reference(V, lab_window, lp_ref, w, e, et, off, reg.n)
    _compare(ph, post, sums, stats, X_own, ref_post, ref_costs, msg)
    return kind


def _expect(D, K, W, s_bound, grid, n, sms, potts=True):
    if bulk_supported(D, K, W, s_bound, potts):
        return "bulk", bulk_instantiation(D, K, grid)
    return "general", general_plan(D, K, n, sms)["n_pass"]


# ---------------------------------------------------------------------------------------------------------------
# (b) every pipeline instantiation
# ---------------------------------------------------------------------------------------------------------------
RAN = set()
B_SMALL = 44            # 990 nodes: 30 full tiles and one of 30 nodes


@pytest.mark.parametrize("D", range(1, 13))
def test_every_bulk_instantiation(ph, sms, calibrated, D):
    from phylo_hmrf_b200 import synth
    rng = np.random.default_rng(100 + D)
    g = synth.make_band(100 + D, B_SMALL, D)
    X, e, w = g["X_own"], g["edge_ids"], g["edge_w"]
    n = len(X)
    assert n % 32 != 0
    W = int(np.bincount(e.ravel()).max())
    i = 0
    for D_, k8 in BULK_PAIRS:
        if D_ != D:
            continue
        for kr in (2, 4, 6, 8):
            for K in (8 * (k8 - 1) + kr - 1, 8 * (k8 - 1) + kr):
                if K < 1:
                    continue
                means, covars = synth.model(200 + K, X, K, D)
                V = synth.potts(K, 0.9)
                lp_ref = orc.compute_log_likelihood(X, means, covars)
                lab = rng.integers(0, K, size=n)
                m = ph.Model(K, D)
                m.set_model(means, covars, V)
                for grid in (False, True):
                    et = 3 if i % 2 == 0 else 0
                    i += 1
                    if grid:
                        reg = m.region_grid(X, 1, B_SMALL, B_SMALL)
                        ee, ww = reg.edges()
                        Wr = 8
                    else:
                        reg = m.region(X, e, w)
                        ee, ww, Wr = e, w, W
                    s_bound = 0.9 * Wr * (np.abs(ww).max() if et == 3 else 1.0)
                    inst = bulk_instantiation(D, K, grid)
                    assert bulk_supported(D, K, Wr, s_bound) and inst[3] == grid and inst[4] == kr
                    _run_case(ph, m, reg, X, lab, ee, ww, V, et, lp_ref, Wr, ("bulk", inst),
                              f"D={D} K={K} grid={grid} et={et}")
                    RAN.add(inst)
                    reg.close()
                m.close()


def test_instantiations_listed(ph):
    ran_d = {t[0] for t in RAN}
    if ran_d != set(range(1, 13)):
        pytest.skip("needs every test_every_bulk_instantiation case in the same session")
    print("\nestep_bulk_kernel<D, NK8, P, GRID, KR> compared with the oracle (%d):" % len(RAN))
    for t in sorted(RAN):
        print("  <%d,%d,%d,%s,%d>" % (t[0], t[1], t[2], "true" if t[3] else "false", t[4]))
    assert RAN == ALL_INSTANTIATIONS


# ---------------------------------------------------------------------------------------------------------------
# (c) routing limits, each just inside and just outside
# ---------------------------------------------------------------------------------------------------------------
def _explicit_case(ph, sms, d, K, V, et, e=None, w=None, seed=0, B=40, label_fn=None):
    X, e0, w0, means, covars = _band_data(seed, B, d, K)
    e = e0 if e is None else e
    w = w0 if w is None else w
    n = len(X)
    W = int(np.bincount(e.ravel(), minlength=n).max())
    potts = np.all(V == V[0, 1] * (1 - np.eye(K))) and V[0, 1] >= 0 if K > 1 else True
    beta = V[0, 1] if K > 1 else 0.0
    s_bound = beta * W * (np.abs(w).max() if et == 3 else 1.0)
    expect = _expect(d, K, W, s_bound, False, n, sms, potts)
    lp_ref = orc.compute_log_likelihood(X, means, covars)
    lab = np.random.default_rng(seed).integers(0, K, size=n) if label_fn is None else label_fn(lp_ref)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    reg = m.region(X, e, w)
    kind = _run_case(ph, m, reg, X, lab, e, w, V, et, lp_ref, W, expect, f"d={d} K={K} W={W} s={s_bound:.3f}")
    reg.close()
    m.close()
    return kind


@pytest.mark.parametrize("d,K_in", [(4, 40), (9, 32), (10, 24), (11, 24), (12, 16)])
def test_state_and_tile_limits(ph, sms, calibrated, d, K_in):
    """K <= 40 and the consumer's accumulator tiles: the last K of the pipeline and the first K past it."""
    from phylo_hmrf_b200 import synth
    for K, want in ((K_in, "bulk"), (K_in + 1, "general")):
        assert _explicit_case(ph, sms, d, K, synth.potts(K, 1.0), 3, seed=K) == want


def test_degree_limit(ph, sms, calibrated):
    """Eight neighbour slots run the pipeline, nine the general kernel."""
    from phylo_hmrf_b200 import synth
    X, e, w, _, _ = _band_data(5, 40, 5, 9)
    deg = np.bincount(e.ravel(), minlength=len(X))
    assert deg.max() == 8
    # one more edge between two nodes of degree 8 that are not yet joined
    have = set(map(tuple, e))
    full = np.flatnonzero(deg == 8)
    a, b = next((int(p), int(q)) for p in full for q in full if p < q and (p, q) not in have)
    e2 = np.concatenate([e, [[a, b]]])
    w2 = np.concatenate([w, [0.5]])
    order = np.lexsort((e2[:, 1], e2[:, 0]))
    assert _explicit_case(ph, sms, 5, 9, synth.potts(9, 1.0), 3, e, w, seed=5) == "bulk"
    assert _explicit_case(ph, sms, 5, 9, synth.potts(9, 1.0), 3, e2[order], w2[order], seed=5) == "general"


@pytest.mark.parametrize("et", [3, 0])
def test_coupling_limit(ph, sms, calibrated, et):
    """|beta| * W * max|w| = 99 runs the pipeline, 101 the general kernel (one edge of weight exactly 1)."""
    from phylo_hmrf_b200 import synth
    X, e, w, _, _ = _band_data(6, 40, 4, 7)
    w = w.copy()
    w[0] = 1.0
    W = int(np.bincount(e.ravel()).max())
    for s, want in ((99.0, "bulk"), (101.0, "general")):
        assert _explicit_case(ph, sms, 4, 7, synth.potts(7, s / W), et, e, w, seed=6) == want


def test_largest_coupling_the_pipeline_takes(ph, sms, calibrated):
    """s_bound = 99.9 with every neighbour on the node's arg-max state and the node labelled at its arg-min, 650 nats
    below: the pipeline's largest soft-max term is about exp(598 + 99.9) -- the overflow-free claim of the kernel."""
    from phylo_hmrf_b200 import synth
    rng = np.random.default_rng(7)
    n, K, d = 997, 5, 3
    # bipartite graph, even ids to odd ids at distance 1, 3, 5, 7: degree 8 inside, so the two colours can disagree
    a = np.arange(0, n, 2)
    e = np.concatenate([np.stack([a, a + s], 1) for s in (1, 3, 5, 7)] + [np.stack([a - s, a], 1) for s in (1, 3, 5, 7)])
    e = e[(e[:, 0] >= 0) & (e[:, 1] < n)]
    e = np.sort(e, axis=1)
    e = np.unique(e, axis=0)
    w = np.ones(len(e))
    W = int(np.bincount(e.ravel()).max())
    assert W == 8
    beta = 99.9 / W
    V = synth.potts(K, beta)
    colour = np.arange(n) % 2
    best = 1 - colour                        # arg-max state: the other colour's label
    lab = colour                             # every node's label: its arg-min
    lp = -300.0 - 300.0 * rng.random((n, K))
    lp[np.arange(n), best] = -2.0 * rng.random(n)
    lp[np.arange(n), lab] = -650.0 - rng.random(n)
    assert np.all(lp.max(1) - lp[np.arange(n), lab] > 600)
    X = _features(rng, n, d)
    means, covars = synth.model(7, X, K, d)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    for et in (3, 0):
        assert bulk_supported(d, K, W, beta * W)
        reg = m.region(X, e, w)
        _run_case(ph, m, reg, X, lab, e, w, V, et, lp, W, ("bulk", None), f"et={et}", set_lp=lp)
        reg.close()
    m.close()


# ---------------------------------------------------------------------------------------------------------------
# (d) several rounds per producer warp, ragged last round
# ---------------------------------------------------------------------------------------------------------------
MULTI = [(2, 3), (9, 30), (11, 20), (12, 16)]     # P = 12 small tile, P = 12 large tile, P = 8, P = 4


def _multi_round_ok(D, K, n, sms):
    P, grid, n_tiles = bulk_launch(D, K, n, sms)
    per = n_tiles // (grid * P)
    rag = n_tiles % (grid * P)
    return grid == sms and per >= 3 and rag != 0 and rag % 4 != 0 and n % 32 != 0


def _assert_multi_round(D, K, n, sms):
    P, grid, n_tiles = bulk_launch(D, K, n, sms)
    assert grid == sms and n_tiles // (grid * P) >= 3, "every producer of every CTA runs three tiles or more"
    assert n_tiles % (grid * P) != 0 and (n_tiles % (grid * P)) % 4 != 0, "ragged last round"
    assert n % 32 != 0


def _n_multi(D, K, sms, extra_tiles=13):
    P = bulk_producers(D, nk8(K))
    n = 32 * (3 * sms * P + extra_tiles) - 5
    assert _multi_round_ok(D, K, n, sms)
    return n


def _tri_start(B, x):
    return x * B - (x * (x - 1)) // 2


def test_multi_round_table():
    """The shapes below cover what they are meant to at 148 SMs (the B200): P and accumulator size."""
    assert [(bulk_producers(D, nk8(K)), bulk_small_acc(D, K)) for D, K in MULTI] == \
        [(12, True), (12, False), (8, False), (4, False)]


@pytest.mark.parametrize("D,K", MULTI)
@pytest.mark.parametrize("layout", ["explicit", "explicit_band", "triangle_band", "rectangle"])
def test_multi_round_pipeline(ph, sms, calibrated, D, K, layout):
    from phylo_hmrf_b200 import synth
    rng = np.random.default_rng(D * 100 + K)
    V = synth.potts(K, 1.0)
    et = 3 if layout in ("explicit", "triangle_band") else 0
    if layout == "explicit":
        n = _n_multi(D, K, sms)
        X = _features(rng, n, D)
        e, w = _rect_edges(n, 517, rng)
        Xw, off = X, 0
    elif layout == "explicit_band":
        n2 = 601
        n = _n_multi(D, K, sms)
        n_window = n + 2 * n2 + 11                 # a halo row above, a row and 11 nodes below
        off = n2
        Xw = _features(rng, n_window, D)
        e, w = _rect_edges(n_window, n2, rng, off, off + n)
        X = Xw[off:off + n]
    elif layout == "triangle_band":
        B = 2400
        r0 = 3
        r1 = next(r for r in range(r0 + 1, B) if _multi_round_ok(D, K, _tri_start(B, r) - _tri_start(B, r0), sms))
        g = synth.window_xy(B, r0, r1)
        Xw = synth.features(D * 7 + K, g["x"], g["y"], D)
        off, n = g["own_offset"], g["n_own"]
        X = Xw[off:off + n]
    else:
        n1 = next(r for r in range(100, 5000) if _multi_round_ok(D, K, r * 389, sms))
        n2 = 389
        n = n1 * n2
        Xw = _features(rng, n, D)
        X, off = Xw, 0
    _assert_multi_round(D, K, n, sms)
    means, covars = synth.model(D + K, X, K, D)
    m = ph.Model(K, D)
    m.set_model(means, covars, V)
    if layout == "explicit":
        reg = m.region(X, e, w)
    elif layout == "explicit_band":
        reg = m.region(X, e, w, n_window=len(Xw), own_offset=off)
    elif layout == "triangle_band":
        reg = m.region_grid(Xw, 1, B, B, r0, r1)
    else:
        reg = m.region_grid(Xw, 0, n1, n2)
    if layout in ("triangle_band", "rectangle"):
        e, w = reg.edges()
        W = 8
    else:
        deg = np.zeros(len(Xw), dtype=np.int64)
        np.add.at(deg, e[:, 0], 1)
        np.add.at(deg, e[:, 1], 1)
        W = int(deg[off:off + n].max())
    assert (reg.n, reg.own_offset) == (n, off)
    lab = rng.integers(0, K, size=len(Xw))
    lp_ref = orc.compute_log_likelihood(X, means, covars)
    grid = layout in ("triangle_band", "rectangle")
    assert bulk_supported(D, K, W, 1.0 * W * (np.abs(w).max() if et == 3 else 1.0))
    _run_case(ph, m, reg, X, lab, e, w, V, et, lp_ref, W, ("bulk", bulk_instantiation(D, K, grid)),
              f"{layout} D={D} K={K} n={n}")
    reg.close()
    m.close()


# whole triangles whose long rows the producers cross with the row walk (rows longer than SMs*P*32/48 nodes)
# and whose short rows near the tip need the closed-form relocation
ROW_WALK = [(2, 3, 1300), (11, 20, 1000), (12, 16, 800)]


@pytest.mark.parametrize("D,K,B0", ROW_WALK)
def test_multi_round_triangle_row_walk(ph, sms, calibrated, D, K, B0):
    from phylo_hmrf_b200 import synth
    P = bulk_producers(D, nk8(K))
    B = next(b for b in range(B0, B0 + 400) if _multi_round_ok(D, K, b * (b + 1) // 2, sms))
    n = B * (B + 1) // 2
    _assert_multi_round(D, K, n, sms)
    step = sms * P * 32
    assert B - 1 > step / 48, "the longest rows are crossed by the row walk"
    g = synth.window_xy(B)
    X = synth.features(D * 11 + K, g["x"], g["y"], D)
    means, covars = synth.model(D * 3 + K, X[::7], K, D)
    V = synth.potts(K, 1.0)
    m = ph.Model(K, D)
    m.set_model(means, covars, V)
    reg = m.region_grid(X, 1, B, B)
    e, w = reg.edges()
    lab = np.random.default_rng(B).integers(0, K, size=n)
    lp_ref = orc.compute_log_likelihood(X, means, covars)
    _run_case(ph, m, reg, X, lab, e, w, V, 3, lp_ref, 8, ("bulk", bulk_instantiation(D, K, True)),
              f"triangle B={B} D={D} K={K}")
    reg.close()
    m.close()


# ---------------------------------------------------------------------------------------------------------------
# (e) general kernel: passes, non-Potts, pairwise potential, striding warps
# ---------------------------------------------------------------------------------------------------------------
PASSES = [(1, 600), (4, 200), (6, 130), (9, 95), (12, 50)]


def test_pass_table():
    for d, K in PASSES:
        p = general_plan(d, K, 1000, 148)
        assert p["n_pass"] >= 3 and p["nkt_total"] % p["nkt_pass"] != 0, (d, K, p)


@pytest.mark.parametrize("d,K", PASSES)
def test_general_kernel_passes(ph, sms, calibrated, d, K):
    from phylo_hmrf_b200 import synth
    p = general_plan(d, K, 990, sms)
    assert p["n_pass"] >= 3 and p["nkt_total"] % p["nkt_pass"] != 0
    for et in (3, 0):
        assert _explicit_case(ph, sms, d, K, synth.potts(K, 0.8), et, seed=d * 1000 + K, B=44) == "general"


def test_general_multipass_non_potts(ph, sms, calibrated):
    d, K = 9, 95
    rng = np.random.default_rng(95)
    V = rng.random((K, K))
    V = 0.5 * (V + V.T)
    np.fill_diagonal(V, 0.0)
    V[0, 1] = V[1, 0] = 0.3
    assert general_plan(d, K, 990, sms)["n_pass"] >= 3
    for et in (3, 0):
        assert _explicit_case(ph, sms, d, K, V, et, seed=95, B=44) == "general"


def test_general_multipass_pairwise_potential(ph, sms, calibrated):
    from phylo_hmrf_b200 import synth
    d, K = 12, 50
    X, e, w, means, covars = _band_data(12, 44, d, K)
    assert general_plan(d, K, len(X), sms)["n_pass"] >= 3
    V = synth.potts(K, 0.7)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    reg = m.region(X, e, w)
    reg.emit_loglik()
    lab = np.random.default_rng(12).integers(0, K, size=len(X))
    reg.set_labels(lab)
    for et in (3, 0):
        pp = reg.pairwise_potential(et)
        np.testing.assert_allclose(pp, orc.pairwise_compare_vec(V, lab, w, e, et), rtol=RTOL, atol=1e-12)
    reg.close()
    m.close()


def test_general_warps_stride_over_three_tiles(ph, sms, calibrated):
    from phylo_hmrf_b200 import synth
    d, K = 4, 200
    p0 = general_plan(d, K, 10 ** 7, sms)
    n = 32 * (3 * sms * p0["wpb"] + 5) - 3
    p = general_plan(d, K, n, sms)
    assert p["grid"] == sms and p["n_tiles"] >= 3 * p["grid"] * p["wpb"] and p["n_pass"] >= 3
    rng = np.random.default_rng(4200)
    X = _features(rng, n, d)
    e, w = _rect_edges(n, 211, rng)
    means, covars = synth.model(4200, X, K, d)
    V = synth.potts(K, 0.6)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    reg = m.region(X, e, w)
    lab = rng.integers(0, K, size=n)
    _run_case(ph, m, reg, X, lab, e, w, V, 3, orc.compute_log_likelihood(X, means, covars), 8,
              ("general", p["n_pass"]), f"d={d} K={K} n={n}")
    reg.close()
    m.close()


# ---------------------------------------------------------------------------------------------------------------
# (f) log-likelihoods far below zero
# ---------------------------------------------------------------------------------------------------------------
LOW = (-1e6 + 30, -1e6 - 5, -1e6 - 650, -2e6)
LOW_SHAPES = [(3, 5), (3, 6), (3, 45), (3, 44)]     # pipeline odd / even K, general odd / even K


@pytest.mark.parametrize("d,K", LOW_SHAPES)
def test_low_loglik_uploaded(ph, sms, calibrated, d, K):
    """Some nodes' best log-likelihood at -1e6 + 30, -1e6 - 5, -1e6 - 650 and -2e6, labelled at the arg-max and away
    from it: the soft-max follows the row maximum, and no state outside 0..K-1 carries weight."""
    from phylo_hmrf_b200 import synth
    X, e, w, means, covars = _band_data(40 + K, 44, d, K)
    n = len(X)
    rng = np.random.default_rng(K)
    lp = -60.0 * rng.random((n, K))
    lab = rng.integers(0, K, size=n)
    rows = rng.choice(n, size=8 * len(LOW), replace=False).reshape(len(LOW), 8)
    for t, rr in zip(LOW, rows):
        for j, i in enumerate(rr):
            lp[i] = t - 40.0 * rng.random(K)
            best = int(rng.integers(K))
            lp[i, best] = t
            lab[i] = best if j % 2 == 0 else (best + 1 + int(rng.integers(K - 1))) % K
    W = int(np.bincount(e.ravel()).max())
    V = synth.potts(K, 1.0)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    for et in (3, 0):
        expect = _expect(d, K, W, 1.0 * W * (np.abs(w).max() if et == 3 else 1.0), False, n, sms)
        reg = m.region(X, e, w)
        _run_case(ph, m, reg, X, lab, e, w, V, et, lp, W, expect, f"K={K} et={et} {expect[0]}", set_lp=lp)
        reg.close()
    m.close()


@pytest.mark.parametrize("K", [5, 6, 45, 44])
def test_low_loglik_emitted(ph, sms, calibrated, K):
    """The same through emission: outlier nodes under tight covariances (d = 9, sigma^2 = 1e-4), about 5 per feature
    from their nearest mean, put the best log-likelihood near -1e6 and below."""
    from phylo_hmrf_b200 import synth
    d, var = 9, 1e-4
    X0, e, w, _, _ = _band_data(50 + K, 44, d, K)
    n = len(X0)
    rng = np.random.default_rng(50 + K)
    means = np.zeros((K, d))
    means[:, 0] = 10.0 * np.arange(K)
    means[:, 1:] = rng.random((K, d - 1))
    covars = np.stack([var * np.eye(d)] * K)
    c = -0.5 * d * np.log(2 * np.pi) - 0.5 * d * np.log(var)    # log-likelihood at the mean
    near = rng.integers(0, K, size=n)
    X = means[near] + 0.004 * rng.standard_normal((n, d))
    rows = rng.choice(n, size=6 * len(LOW), replace=False).reshape(len(LOW), 6)
    for t, rr in zip(LOW, rows):
        r2 = 2.0 * var * (c - t)                                # squared distance to the nearest mean
        v = -np.ones(d) * np.sqrt(r2 / d)                       # away from the other means (feature 0 decreases)
        X[rr] = means[0] + v
        near[rr] = 0
    lab = near.copy()
    lab[::3] = (lab[::3] + 1) % K                               # a third labelled away from the nearest mean
    W = int(np.bincount(e.ravel()).max())
    V = synth.potts(K, 1.0)
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    reg = m.region(X, e, w)
    reg.emit_loglik()
    lp = reg.logprob()
    lp_ref = orc.compute_log_likelihood(X, means, covars)
    np.testing.assert_allclose(lp, lp_ref, rtol=1e-10)
    for t, rr in zip(LOW, rows):
        np.testing.assert_allclose(lp[rr].max(axis=1), t, rtol=1e-10)
    reg.close()
    for et in (3, 0):
        reg = m.region(X, e, w)
        expect = _expect(d, K, W, 1.0 * W * (np.abs(w).max() if et == 3 else 1.0), False, n, sms)
        # the E-step is compared on the library's own log-likelihood (equal to the oracle's to 1e-10 above)
        _run_case(ph, m, reg, X, lab, e, w, V, et, lp, W, expect, f"K={K} et={et} {expect[0]}")
        reg.close()
    m.close()
