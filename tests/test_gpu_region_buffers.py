"""What a region holds on the device, written out buffer by buffer: phmrf_region_device_bytes for both region
kinds, fresh and after the E-step and graph cut grow them, the kernels that building a region launches, and
regions built and closed in a loop."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
K, D = 10, 4


@pytest.fixture(scope="module")
def ph():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import phylo_hmrf_b200 as ph
    return ph


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def model(ph):
    from phylo_hmrf_b200 import synth
    means, covars = synth.model(5, synth.make_band(5, 40, D)["X_own"], K, D)
    m = ph.Model(K, D)
    m.set_model(means, covars, synth.potts(K, 1.0))
    yield m
    m.close()


def _round_up(x, m):
    return -(-x // m) * m


def _shared_bytes(sm, n_own, n_window, W, E):
    """The buffers both region kinds allocate; an element count below one allocates one element."""
    one = lambda c: max(c, 1)
    ld = _round_up(max(n_own, 1), 64)
    rows = _round_up(K, 8)                        # log-likelihood rows (common.cuh logp_rows)
    F = 1 + D + D * (D + 1) // 2                  # statistics features per state
    stats_len = K * (1 + D + D * D) + 3
    return (8 * D * ld                            # X
            + 8 * rows * ld                       # log-likelihood
            + 8 * ld                              # per-node maximum
            + 4 * one(n_own * K)                  # integer unary
            + 4 * one(n_window)                   # labels
            + 4 * one(W * ld) + 8 * one(W * ld)   # neighbour ids and weights
            + 8 * one(E) + 4 * one(E)             # edge weights, integer edge weights
            + 8 * 2 + 8 * 2                       # absmax / boundary counter, dwf
            + 8 * (1 << 20)                       # boundary list
            + 8 * sm * (K * F + 3)                # per-CTA partial sums
            + 8 * stats_len + 4 + 8)              # statistics, overflow flag, first bad label


def _general_bytes(sm, n, W, E):
    return _shared_bytes(sm, n, n, W, E) + 8 * n * D     # + the scratch that staged X


def _grid_bytes(sm, n_own, n_window, own_offset, E):
    ldw = _round_up(own_offset + n_own, 64)
    return _shared_bytes(sm, n_own, n_window, 8, E) + 8 * max(2 * E, 1) + 16 * 4 * ldw  # + edge ids, forward weights


def _cut_bytes(n, E):
    """swap_scratch_alloc: 52 bytes per site, 36 per slot (2E slots), V and the fixed words."""
    return 52 * n + 36 * 2 * E + 3 * 8 + 4 * K * K + 8 * 8


def _max_degree(edge_ids, n):
    return int(np.bincount(edge_ids.ravel(), minlength=n).max())


def _general(ph, m, B=40, seed=5):
    from phylo_hmrf_b200 import synth
    g = synth.make_band(seed, B, D)
    c0 = ph.engine.launch_count()
    r = m.region(g["X_own"], g["edge_ids"], g["edge_w"])
    return r, g, ph.engine.launch_count() - c0


def _grid(ph, m, B=40, rows=None, seed=5):
    from phylo_hmrf_b200 import synth
    r0, r1 = rows or (0, B)
    g = synth.make_band(seed, B, D, r0, r1, beta1=0.1)
    c0 = ph.engine.launch_count()
    r = m.region_grid(g["X_window"], 1, B, B, r0, r1, num_neighbor=8, beta1=0.1)
    return r, g, ph.engine.launch_count() - c0


def test_general_region_bytes(ph, model, sm_count):
    r, g, launches = _general(ph, model)
    try:
        n, E = r.n, r.n_edges
        W = _max_degree(g["edge_ids"], n)
        ld = _round_up(n, 64)
        assert launches == 2                                   # log-likelihood init, X transpose
        expect = _general_bytes(sm_count, n, W, E)
        assert r.device_bytes() == expect
        r.emit_loglik()
        r.set_labels(np.random.default_rng(0).integers(0, K, n).astype(np.int32))
        r.estep_stats(3)                                       # the pipeline kernel's per-slot factors
        expect += 8 * W * ld
        assert r.device_bytes() == expect
        r.estep_stats(3, want_post=True)                       # the scratch grows to [K][ld] + [n,K]
        expect += 8 * (K * ld + n * K) - 8 * n * D
        assert r.device_bytes() == expect
    finally:
        r.close()


@pytest.mark.parametrize("rows", [None, (13, 27)])
def test_grid_region_and_band_bytes(ph, model, sm_count, rows):
    r, g, launches = _grid(ph, model, rows=rows)
    try:
        assert (r.n, r.n_window, r.own_offset) == (g["n_own"], len(g["X_window"]), g["own_offset"])
        assert r.n_edges == len(g["edge_ids"])
        # edge counting (2), log-likelihood init, X transpose, forward weights, edge list and neighbour slots (4)
        assert launches == 9
        assert r.device_bytes() == _grid_bytes(sm_count, r.n, r.n_window, r.own_offset, r.n_edges)
    finally:
        r.close()


def test_grid_region_bytes_after_the_first_cut(ph, model, sm_count):
    r, g, _ = _grid(ph, model)
    try:
        fresh = _grid_bytes(sm_count, r.n, r.n_window, r.own_offset, r.n_edges)
        r.emit_loglik()
        q = r.quantise()
        r.graph_cut(np.argmin(q["unary_i32"], axis=1).astype(np.int32), n_iter=5)
        assert r.device_bytes() == fresh + _cut_bytes(r.n, r.n_edges)
        r.graph_cut(None, n_iter=2)                            # the second cut reuses the scratch
        assert r.device_bytes() == fresh + _cut_bytes(r.n, r.n_edges)
    finally:
        r.close()


def test_regions_built_cut_and_closed_in_a_loop(ph, model):
    first = {}
    for i in range(20):
        for kind, make in (("general", _general), ("grid", _grid)):
            r, _, _ = make(ph, model)
            try:
                first.setdefault(kind, r.device_bytes())
                assert r.device_bytes() == first[kind], (kind, i)
                r.emit_loglik()
                q = r.quantise(want_edges=False)
                r.graph_cut(np.argmin(q["unary_i32"], axis=1).astype(np.int32), n_iter=2)
                r.estep_stats(3)
            finally:
                r.close()
