"""NumPy reference of the per-node posterior summary (phmrf_posterior_summary), built on the vectorised
posteriors of oracle/phmrf_oracle.py: pp from pairwise_compare_vec over the label window, the max-shifted
soft-max of logp - pp."""
import numpy as np

from oracle import phmrf_oracle as orc


def summary_from_logits(a, labels):
    """Summary of the posteriors softmax(a) [n,K] at labels [n]."""
    a = np.asarray(a, dtype=np.float64)
    n = len(a)
    post = orc._stable_softmax(a)
    m = a.max(axis=1, keepdims=True)
    z = np.exp(a - m)
    Z = z.sum(axis=1)
    t = np.where(z > 0, z * (a - m), 0.0).sum(axis=1)
    ms = np.argmax(post, axis=1).astype(np.int32)
    rows = np.arange(n)
    return dict(map_state=ms, map_prob=post[rows, ms], label_prob=post[rows, np.asarray(labels, dtype=np.int64)],
                entropy=np.log(Z) - t / Z)


def summary(V, labels_window, logp, edge_w, edge_ids, estimate_type, own_offset=0):
    """Summary of the owned rows [own_offset, own_offset + len(logp)) of a label window."""
    lab = np.asarray(labels_window, dtype=np.int64)
    n = len(logp)
    pp = orc.pairwise_compare_vec(V, lab, edge_w, edge_ids, estimate_type)[own_offset:own_offset + n]
    return summary_from_logits(np.asarray(logp) - pp, lab[own_offset:own_offset + n])


def assert_summary_close(got, ref, rtol=1e-9, atol_entropy=1e-12):
    np.testing.assert_array_equal(got["map_state"], ref["map_state"])
    np.testing.assert_allclose(got["map_prob"], ref["map_prob"], rtol=rtol, atol=0)
    np.testing.assert_allclose(got["label_prob"], ref["label_prob"], rtol=rtol, atol=1e-300)
    np.testing.assert_allclose(got["entropy"], ref["entropy"], rtol=0, atol=atol_entropy)
