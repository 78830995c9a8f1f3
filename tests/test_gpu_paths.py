"""Every phase-B code path against the oracle: the DMMA pipeline (Potts, <=8 slots, K<=40), and
the general kernel it defers to (K>40 multi-pass, degree>8 graphs, strong coupling
beta*W*max|w| >= 100, non-Potts V), plus labels far from the arg-max (soft-max shift)."""
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


def _check(ph, X, e, w, means, covars, V, lab, et, rtol=RTOL, general=False):
    """general: the shape runs the general kernel, which reads the neighbour ids and weights only, so an
    E-step must not allocate the pipeline's per-slot factor array (without posteriors nothing else grows)."""
    K, d = means.shape
    m = ph.Model(K, d)
    m.set_model(means, covars, V)
    reg = m.region(X, e, w)
    reg.emit_loglik()
    lp_ref = orc.compute_log_likelihood(X, means, covars)
    reg.set_labels(lab)
    if general:
        before = reg.device_bytes()
        reg.estep_stats(et)
        assert reg.device_bytes() == before
    stats, sums, post = reg.estep_stats(et, want_post=True)
    ref = orc.compute_posteriors_graph(V, lab, lp_ref, w, e, None, et, faithful=False, stable=True)
    np.testing.assert_allclose(post, ref[0], rtol=rtol, atol=1e-290)
    np.testing.assert_allclose(ph.costs_from_sums(sums, len(X)), ref[1:], rtol=rtol, atol=1e-12)
    st = orc.sufficient_statistics(ref[0], X)
    for key in st:
        np.testing.assert_allclose(stats[key], st[key], rtol=rtol, atol=rtol * 1e-3 * np.abs(st[key]).max())
    reg.close()
    m.close()


def _data(seed, B, d, K):
    from phylo_hmrf_b200 import synth
    g = synth.make_band(seed, B, d)
    means, covars = synth.model(seed, g["X_own"], K, d)
    return g["X_own"], g["edge_ids"], g["edge_w"], means, covars


def test_more_than_40_states_general_multipass(ph):
    # d = 9: one pass of the general kernel holds 6 k-tiles of 5 states, so K = 45 takes two passes
    from phylo_hmrf_b200 import synth
    X, e, w, means, covars = _data(1, 45, 9, 45)
    lab = np.random.default_rng(1).integers(0, 45, size=len(X))
    _check(ph, X, e, w, means, covars, synth.potts(45, 1.0), lab, 3, general=True)


def test_degree_above_eight_general_graph(ph):
    from phylo_hmrf_b200 import synth
    X, e, w, means, covars = _data(2, 30, 4, 7)
    rng = np.random.default_rng(2)
    n = len(X)
    extra = np.sort(rng.integers(0, n, size=(600, 2)), axis=1)  # long-range edges: degrees up to ~14
    extra = extra[extra[:, 0] != extra[:, 1]]
    have = set(map(tuple, e))
    extra = np.array([p for p in map(tuple, extra) if p not in have])
    extra = np.unique(extra, axis=0)
    e2 = np.concatenate([e, extra])
    w2 = np.concatenate([w, rng.random(len(extra))])
    order = np.lexsort((e2[:, 1], e2[:, 0]))
    e2, w2 = e2[order], w2[order]
    deg = np.bincount(e2.ravel(), minlength=n)
    assert deg.max() > 8
    _check(ph, X, e2, w2, means, covars, synth.potts(7, 0.8), rng.integers(0, 7, size=n), 3, general=True)


def test_strong_coupling_routes_to_exact_path(ph):
    from phylo_hmrf_b200 import synth
    X, e, w, means, covars = _data(3, 28, 5, 9)
    lab = np.random.default_rng(3).integers(0, 9, size=len(X))
    _check(ph, X, e, w, means, covars, synth.potts(9, 40.0), lab, 3, general=True)     # beta*8*max(w) >= 100
    _check(ph, X, e, w, means, covars, synth.potts(9, 40.0), lab, 0, general=True)


def test_labels_far_from_the_argmax(ph):
    """Tight covariances make the log-likelihood gaps exceed 700 nats: the soft-max shift must
    follow the row maximum, not the (bad) label."""
    from phylo_hmrf_b200 import synth
    X, e, w, means, _ = _data(4, 33, 9, 30)
    covars = np.stack([2e-3 * np.eye(9)] * 30)
    lp = orc.compute_log_likelihood(X, means, covars)
    worst = np.argmin(lp, axis=1)
    assert (lp.max(axis=1) - lp[np.arange(len(X)), worst]).max() > 2000
    _check(ph, X, e, w, means, covars, synth.potts(30, 1.0), worst, 3)
    _check(ph, X, e, w, means, covars, synth.potts(30, 1.0), np.argmax(lp, axis=1), 3)


@pytest.mark.parametrize("d,K", [(1, 2), (2, 8), (3, 9), (4, 16), (5, 20), (6, 24), (7, 5), (8, 33), (10, 12), (11, 6),
                                 (12, 3), (12, 30)])
def test_every_feature_count_and_state_tiling(ph, d, K):
    from phylo_hmrf_b200 import synth
    X, e, w, means, covars = _data(10 + d, 26, d, K)
    lab = np.random.default_rng(d).integers(0, K, size=len(X))
    # d = 12, K = 30: the 4 x 12 accumulator tiles do not fit the pipeline's consumer registers
    _check(ph, X, e, w, means, covars, synth.potts(K, 1.0), lab, 3, general=(d, K) == (12, 30))


def test_slot_factor_cache_follows_beta_and_weighting(ph):
    """The pipeline keeps exp(beta*w) per neighbour slot on the device between E-steps of one
    region: a new beta (set_model) or a switch between weighted and unweighted estimates must
    rebuild it."""
    from phylo_hmrf_b200 import synth
    X, e, w, means, covars = _data(11, 30, 5, 12)
    K, d = means.shape
    lab = np.random.default_rng(11).integers(0, K, size=len(X))
    lp_ref = orc.compute_log_likelihood(X, means, covars)
    m = ph.Model(K, d)
    m.set_model(means, covars, synth.potts(K, 0.7))
    reg = m.region(X, e, w)
    reg.emit_loglik()
    reg.set_labels(lab)
    for beta, et in ((0.7, 3), (0.7, 0), (1.9, 0), (1.9, 3), (0.7, 3)):
        V = synth.potts(K, beta)
        m.set_model(means, covars, V)
        reg.emit_loglik()
        stats, sums, post = reg.estep_stats(et, want_post=True)
        ref = orc.compute_posteriors_graph(V, lab, lp_ref, w, e, None, et, faithful=False, stable=True)
        np.testing.assert_allclose(post, ref[0], rtol=RTOL, atol=1e-290, err_msg=f"beta={beta} et={et}")
        np.testing.assert_allclose(ph.costs_from_sums(sums, len(X)), ref[1:], rtol=RTOL, atol=1e-12)
    reg.close()
    m.close()
