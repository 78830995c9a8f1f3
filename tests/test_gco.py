"""Host graph cut (include/phmrf_gco.h, csrc/gco.cpp): GCO v3.0's general-graph swap and expansion.

Known answers: the six scenarios of GCO's own example program (gco_source/example.cpp of the
reference), 250 -> 44/44/44/170/44/244."""
import itertools

import numpy as np
import pytest


@pytest.fixture(scope="module")
def engine():
    from phylo_hmrf_b200 import build, engine
    build.build_gco()
    return engine


def _example_grid(h_weight, v_weight):
    """example.cpp's 10x5 grid, 7 labels: data 0 for label 0 on the first 25 sites and label 5 on the
    others, 10 otherwise; smooth min((l1-l2)^2, 4); h_weight/v_weight(p1, p2) weigh the horizontal and
    vertical neighbour pairs."""
    width, height, L = 10, 5, 7
    n = width * height
    data = np.full((n, L), 10, dtype=np.int32)
    data[:25, 0] = 0
    data[25:, 5] = 0
    l = np.arange(L)
    smooth = np.minimum((l[:, None] - l[None, :]) ** 2, 4).astype(np.int32)
    e, w = [], []
    for y in range(height):
        for x in range(1, width):
            p1, p2 = x - 1 + y * width, x + y * width
            e.append((p1, p2)); w.append(h_weight(p1, p2))
    for y in range(1, height):
        for x in range(width):
            p1, p2 = x + (y - 1) * width, x + y * width
            e.append((p1, p2)); w.append(v_weight(p1, p2))
    return data, np.asarray(e, dtype=np.int64), np.asarray(w, dtype=np.int32), smooth


def test_gco_example_known_answers(engine):
    """example.cpp runs expansion(2) from the all-zero labelling on six set-ups of three energies:
    grid with unit weights (set individually, by arrays, by functions), grid with spatially varying
    weights H[p] = p+(p+1)%3, V[p] = p*(p+width)%7 (setSmoothCostVH), the grid as a general graph
    with unit weights, and as a general graph with weights p1+p2 (horizontal) and p1*p2 (vertical)."""
    unit = _example_grid(lambda a, b: 1, lambda a, b: 1)
    vh = _example_grid(lambda a, b: a + (a + 1) % 3, lambda a, b: a * (a + 10) % 7)
    spat = _example_grid(lambda a, b: a + b, lambda a, b: a * b)
    before, after = [], []
    for data, e, w, smooth in (unit, unit, unit, vh, unit, spat):
        _, en, en0 = engine.gco_cut_int(data, e, w, smooth, n_iter=2, algorithm='expansion', return_energy=True)
        before.append(en0)
        after.append(en)
    assert before == [250] * 6
    assert after == [44, 44, 44, 170, 44, 244]


def _energy(unary, e, w, V, lab):
    return int(unary[np.arange(len(lab)), lab].sum() + (V[lab[e[:, 0]], lab[e[:, 1]]].astype(np.int64) * w).sum())


def test_wrapper_reproduces_example_energies(engine):
    """GeneralGraph_DArraySArraySpatVarying of example.cpp: the returned labels have the returned energy."""
    data, e, w, smooth = _example_grid(lambda a, b: a + b, lambda a, b: a * b)
    lab, en, en0 = engine.gco_cut_int(data, e, w, smooth, n_iter=2, algorithm='expansion', return_energy=True)
    assert en0 == 250 and en == 244
    assert _energy(data, e, w, smooth, lab) == 244


def test_swap_from_init_labels_is_deterministic_and_monotone(engine):
    rng = np.random.default_rng(5)
    n, K = 60, 5
    unary = rng.integers(0, 1000, size=(n, K)).astype(np.int32)
    e = np.asarray([(i, j) for i in range(n) for j in range(i + 1, min(n, i + 4))], dtype=np.int64)
    w = rng.integers(1, 50, size=len(e)).astype(np.int32)
    V = (30 * (1 - np.eye(K))).astype(np.int32)
    init = rng.integers(0, K, size=n).astype(np.int32)
    lab1, en1, en0 = engine.gco_cut_int(unary, e, w, V, n_iter=5000, algorithm='swap', init_labels=init,
                                        return_energy=True)
    lab2 = engine.gco_cut_int(unary, e, w, V, n_iter=5000, algorithm='swap', init_labels=init)
    assert np.array_equal(lab1, lab2)
    assert en0 == _energy(unary, e, w, V, init)
    assert en1 == _energy(unary, e, w, V, lab1) <= en0
    # a swap-converged labelling is single-site optimal
    for i in range(n):
        for k in range(K):
            trial = lab1.copy(); trial[i] = k
            assert _energy(unary, e, w, V, trial) >= en1


def test_two_label_swap_is_globally_optimal(engine):
    rng = np.random.default_rng(9)
    n = 10
    unary = rng.integers(0, 100, size=(n, 2)).astype(np.int32)
    e = np.asarray([(i, i + 1) for i in range(n - 1)] + [(0, 5), (2, 7)], dtype=np.int64)
    w = rng.integers(1, 40, size=len(e)).astype(np.int32)
    V = np.asarray([[0, 1], [1, 0]], dtype=np.int32)
    lab, en, _ = engine.gco_cut_int(unary, e, w, V, n_iter=100, algorithm='swap',
                                    init_labels=np.zeros(n, np.int32), return_energy=True)
    best = min(_energy(unary, e, w, V, np.asarray(c)) for c in itertools.product((0, 1), repeat=n))
    assert en == best


def test_errors_come_back_as_exceptions_not_exits(engine):
    unary = np.zeros((4, 3), dtype=np.int32)
    V = np.zeros((3, 3), dtype=np.int32)
    with pytest.raises(RuntimeError, match="id1 < id2"):
        engine.gco_cut_int(unary, np.asarray([[2, 1]]), np.asarray([1], np.int32), V, algorithm='swap')
    with pytest.raises(RuntimeError, match="init label"):
        engine.gco_cut_int(unary, np.asarray([[0, 1]]), np.asarray([1], np.int32), V, algorithm='swap',
                           init_labels=np.asarray([0, 1, 2, 3]))
    # a smoothness term beyond GCO_MAX_ENERGYTERM is an error returned to the caller, not a process exit
    big = (5000 * (1 - np.eye(3))).astype(np.int32)
    with pytest.raises(RuntimeError, match="GCO"):
        engine.gco_cut_int(unary, np.asarray([[0, 1]]), np.asarray([20000000], np.int32), big, algorithm='swap',
                           init_labels=np.asarray([0, 1, 2, 0]))
    with pytest.raises(TypeError):
        engine.cut_general_graph(np.asarray([[0, 1]]), np.asarray([0.5]), unary, V, algorithm='swap')


def _moves_by_enumeration(unary, e, w, V, init, n_iter, algorithm):
    """GCO's cycles with every move solved by enumeration: among the minimum-energy assignments of the
    move's binary variables (0 = alpha), a variable is 1 only when it is 1 in all of them -- the cut
    with the smallest sink side, which the max-flow of GCO returns."""
    def energy(lab):
        return int(unary[np.arange(len(lab)), lab].sum() + (V[lab[e[:, 1]], lab[e[:, 0]]].astype(np.int64) * w).sum())

    def move(lab, active, label_of):
        best, argmins = None, []
        for bits in itertools.product((0, 1), repeat=len(active)):
            trial = lab.copy()
            trial[active] = [label_of(b, s) for b, s in zip(bits, active)]
            en = energy(trial)
            if best is None or en < best:
                best, argmins = en, [bits]
            elif en == best:
                argmins.append(bits)
        bits = np.min(np.asarray(argmins), axis=0)
        lab[active] = [label_of(b, s) for b, s in zip(bits, active)]

    K = unary.shape[1]
    lab = init.copy()
    en, old, cycle = energy(lab), energy(lab) + 1, 1
    while old > en and cycle <= n_iter:
        old = en
        if algorithm == 'swap':
            for a in range(K):
                for b in range(K - 1, a, -1):
                    active = np.flatnonzero((lab == a) | (lab == b))
                    if len(active):
                        move(lab, active, lambda x, s, a=a, b=b: a if x == 0 else b)
        else:
            for a in range(K):
                active, cur = np.flatnonzero(lab != a), lab.copy()
                if len(active):
                    move(lab, active, lambda x, s, a=a, cur=cur: a if x == 0 else cur[s])
        en = energy(lab)
        cycle += 1
    return lab, en


@pytest.mark.parametrize("algorithm", ["swap", "expansion"])
def test_labels_follow_the_move_rule_on_ties(engine, algorithm):
    """Small costs make many equal-energy moves; the labels must still be the ones GCO's order of moves
    and choice of cut give, not just some labelling of the same energy."""
    rng = np.random.default_rng(11)
    for _ in range(60):
        n, K = int(rng.integers(2, 10)), int(rng.integers(2, 5))
        e = np.asarray([(i, j) for i in range(n) for j in range(i + 1, n) if rng.random() < 0.35],
                       dtype=np.int64).reshape(-1, 2)
        w = rng.integers(0, 6, len(e)).astype(np.int32)
        unary = rng.integers(0, 8, (n, K)).astype(np.int32)
        if algorithm == 'swap':
            M = rng.integers(0, 4, (K, K))
            V = (M + M.T) * (1 - np.eye(K, dtype=np.int64))
        else:
            V = int(rng.integers(1, 3)) * (1 - np.eye(K, dtype=np.int64))   # Potts: a metric
        V = V.astype(np.int32)
        init = rng.integers(0, K, n).astype(np.int32)
        lab, en, _ = engine.gco_cut_int(unary, e, w, V, n_iter=50, algorithm=algorithm, init_labels=init,
                                        return_energy=True)
        lab_ref, en_ref = _moves_by_enumeration(unary, e, w, V, init, 50, algorithm)
        assert en == en_ref
        assert np.array_equal(lab, lab_ref)


@pytest.mark.parametrize("case", ["b56_k10", "b40_k20"])
def test_pinned_labels_of_quantised_regions(engine, case):
    """The product's call (swap, n_iter=5000, arg-min start) and expansion(2) / expansion(-1) on the integer arrays
    of two quantised regions give the stored labels and energies (tests/golden/make_golden_gco.py: pinned from this
    graph cut, GCO itself not being part of the repository)."""
    import os
    from phylo_hmrf_b200 import synth
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gco_regions.npz"))
    u, w, V = G[case + "_unary"], G[case + "_w"], G[case + "_V"]
    B = int(case[1:case.index("_")])
    e = synth.triangle_band(B, 0, B)["edge_ids"]
    init = np.argmin(u, axis=1).astype(np.int32)
    for alg, n_iter in (("swap", 5000), ("expansion", 2), ("expansion", -1)):
        lab, en, _ = engine.gco_cut_int(u, e, w, V, n_iter=n_iter, algorithm=alg, init_labels=init, return_energy=True)
        key = case + "_%s%d_" % (alg, n_iter)
        assert en == int(G[key + "energy"]) == _energy(u, e, w, V, lab)
        np.testing.assert_array_equal(lab, G[key + "labels"])
