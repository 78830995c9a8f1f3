"""Host cut (csrc/gco.cpp) against the device cut (kernels_cut.cu) on the same integer arrays.

    python tools/bench_graph_cut.py [--out profiles/r3_graph_cut.json] [--host-budget 300] [--shapes ...]

Each shape is a synthetic diagonal region of B bins (B(B+1)/2 nodes, 8 neighbours) built on the device through a
GridRegion, its log-likelihood quantised there, and cut from the arg-min of the integer unary with n_iter=5000
(the product's call).  The device cut runs on the region's own arrays (Region.graph_cut); the host cut on the same
arrays downloaded (quantise + edges).  Times are host wall clocks around calls that end in a device synchronise.
The first device cut of a region also builds its graph and scratch; shapes up to --warm-max nodes are cut a
second time to show the steady-state time.  The host cut runs where its projected time (the last host time scaled
by N*K^2) stays within --host-budget seconds.  Where both ran, the labels and energies must be identical."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from phylo_hmrf_b200 import engine, synth  # noqa: E402

# (name, bins, K): the chr21 example (cfg 1), chr21+chr22 (cfg 2), a 2.0 M-node region, chr1 at 50 kb (cfg 3),
# and about one headline band (38.7 M nodes at K = 30)
SHAPES = [("b652_k10", 652, 10), ("b683_k20", 683, 20), ("b2000_k20", 2000, 20), ("b4979_k20", 4979, 20),
          ("b8800_k30", 8800, 30)]
D = 5


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        return "nvidia-smi unavailable: %s" % ex


def one_shape(name, B, K, host_allowed, warm_max, seed=20261020):
    w = synth.window_xy(B)
    X = synth.features(seed, w["x"], w["y"], D)
    n = len(X)
    means, covars = synth.model(seed, X[:: max(1, n // 200000)], K, D)
    m = engine.Model(K, D)
    m.set_model(means, covars, synth.potts(K, 1.0))
    r = m.region_grid(X, 1, B, B, num_neighbor=8, beta1=0.1)
    del X
    res = dict(shape=name, bins=B, K=K, nodes=n, edges=r.n_edges)
    try:
        r.emit_loglik()
        r.quantise(want_unary=False, want_edges=False)
        init = r.labels_argmin_unary()
        bytes0 = r.device_bytes()
        t0 = time.perf_counter()
        lab_d, en_d, en0 = r.graph_cut(init, n_iter=5000, return_energy=True)
        res["device_s_first"] = time.perf_counter() - t0
        res["device_scratch_bytes"] = r.device_bytes() - bytes0
        res["energy_before"], res["energy_device"] = en0, en_d
        res["labels_changed"] = int(np.count_nonzero(lab_d != init))
        if n <= warm_max:
            t0 = time.perf_counter()
            lab_w = r.graph_cut(init, n_iter=5000)
            res["device_s_warm"] = time.perf_counter() - t0
            assert np.array_equal(lab_w, lab_d)
        # bytes over PCIe per region and EM pass, from the shapes: host mode downloads the integer unary and edge
        # weights and uploads the labels; device mode uploads the init labels and downloads the result
        res["pcie_bytes_host_mode"] = 4 * n * K + 4 * r.n_edges + 4 * n
        res["pcie_bytes_device_mode"] = 4 * n + 4 * n
        if host_allowed:
            q = r.quantise()
            ids, _ = r.edges()
            t0 = time.perf_counter()
            lab_h, en_h, en0_h = engine.gco_cut_int(q["unary_i32"], ids, q["w_i32"], q["V_i32"], n_iter=5000,
                                                    algorithm='swap', init_labels=init, return_energy=True)
            res["host_s"] = time.perf_counter() - t0
            res["energy_host"] = en_h
            res["labels_identical"] = bool(np.array_equal(lab_h, lab_d) and en_h == en_d and en0_h == en0)
            assert res["labels_identical"], "device and host cuts differ on %s" % name
    finally:
        r.close()
        m.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r3_graph_cut.json")
    ap.add_argument("--host-budget", type=float, default=300.0)
    ap.add_argument("--warm-max", type=int, default=2_100_000)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_graph_cut.py measures the GPU cut: no CUDA device")
    out = dict(gpu=gpu_info(), n_iter=5000, start="arg-min of the integer unary", features=D, results=[])
    last = None   # (host seconds, nodes * K^2) of the last host cut
    for name, B, K in SHAPES:
        if name not in a.shapes.split(","):
            continue
        cost = (B * (B + 1) // 2) * K * K
        projected = None if last is None else last[0] * cost / last[1]
        host_allowed = projected is None or projected <= a.host_budget
        res = one_shape(name, B, K, host_allowed, a.warm_max)
        if not host_allowed:
            res["host_skipped"] = "projected %.0f s > budget %.0f s" % (projected, a.host_budget)
        if "host_s" in res:
            last = (res["host_s"], cost)
        out["results"].append(res)
        print(json.dumps(res), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:       # after every shape: the large ones take minutes
            json.dump(out, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
