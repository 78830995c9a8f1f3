"""tests/golden/gco_regions.npz: integer cost arrays of two quantised regions (the edge list
is synth.triangle_band's, rebuilt by the test) and the labels and energies the
graph cut (csrc/gco.cpp) gave for them -- swap with n_iter=5000 from the arg-min of the unary (the product
path), expansion with n_iter=2 and -1 from the same start.  GCO v3.0 itself is not part of this repository,
so these pin the in-tree graph cut against later changes; they were not produced by GCO.

    python tests/golden/make_golden_gco.py      (after python -m phylo_hmrf_b200.build)"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import phmrf_oracle as orc  # noqa: E402
from phylo_hmrf_b200 import engine, synth  # noqa: E402

CASES = {"b56_k10": (20261101, 56, 4, 10), "b40_k20": (20261102, 40, 5, 20)}


def main():
    out = {}
    for name, (seed, B, d, K) in CASES.items():
        g = synth.make_band(seed, B, d, beta1=0.1)
        means, covars = synth.model(seed, g["X_own"], K, d)
        lp = orc.compute_log_likelihood(g["X_own"], means, covars)
        u, w, V, _ = orc.pygco_quantise(-lp, g["edge_w"], synth.potts(K, 1.0))
        init = np.argmin(u, axis=1).astype(np.int32)
        p = name + "_"
        assert np.array_equal(g["edge_ids"], synth.triangle_band(B, 0, B)["edge_ids"])
        out.update({p + "unary": u, p + "w": w, p + "V": V})
        for alg, n_iter in (("swap", 5000), ("expansion", 2), ("expansion", -1)):
            lab, en, _ = engine.gco_cut_int(u, g["edge_ids"], w, V, n_iter=n_iter, algorithm=alg, init_labels=init,
                                            return_energy=True)
            key = p + "%s%d_" % (alg, n_iter)
            out[key + "labels"] = lab.astype(np.int8)
            out[key + "energy"] = np.int64(en)
    np.savez_compressed(os.path.join(HERE, "gco_regions.npz"), **out)


if __name__ == "__main__":
    main()
