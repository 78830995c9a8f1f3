"""Time the posterior-summary kernel (phmrf_posterior_summary) with CUDA events over many launches on two shapes
and report its algorithmic bytes over the measured time against the HBM data-sheet peak.

    python tools/bench_posterior_summary.py [--launches N] [--out file.json]

* ``cfg5_band``: one of the eight row bands of chr1 at 10 kb (B = 24895 bins, band 0: 38.7 M nodes), d = 9,
  K = 30, built on the device from the grid geometry (implicit neighbours) -- the shape bench.py times.
* ``cfg3``: chr1 at 50 kb as one whole region (B = 4979, 12.4 M nodes), d = 5, K = 20, grid-built.

Both working sets are far larger than the 126 MB L2, so every launch reads from HBM.  The E-step of the same
region (phmrf_estep_stats_async) is timed alongside, for the cost of one summary relative to one iteration's
phase B.  Algorithmic bytes per node: 8*KP log-likelihood (KP = K rounded up to 8), 4 for the label, the
neighbour data (grid-built, estimate_type 3: four forward {w, exp(beta*w)} pairs, 64 bytes) and 28 written.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_DATASHEET_GBS = 7700.0   # HGX B200 data sheet, one GPU, at up to 1000 W
SHAPES = {"cfg5_band": dict(B=24895, bands=8, d=9, K=30), "cfg3": dict(B=4979, bands=0, d=5, K=20)}
ET, BETA, BETA1, SEED = 3, 1.0, 0.1, 20261017


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [v.strip() for v in q.split(",")]
        return dict(name=name, power_limit=power, sm_max_clock=clk)
    except Exception as exc:          # the timing stands without it, but say so
        return dict(error=repr(exc))


def time_launches(torch, stream, fn, n):
    for _ in range(3):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        start.record(stream)
        for _ in range(n):
            fn()
        end.record(stream)
    end.synchronize()
    return start.elapsed_time(end) / n


def one_shape(torch, ph, synth, name, launches):
    s = SHAPES[name]
    B, d, K = s["B"], s["d"], s["K"]
    r0, r1 = synth.band_rows(B, s["bands"])[0] if s["bands"] else (0, B)
    g = synth.window_xy(B, r0, r1)
    X = synth.features(SEED, g["x"], g["y"], d)
    g.clear()
    means, covars = synth.model(SEED, X[:200000], K, d)
    m = ph.Model(K, d)
    m.set_model(means, covars, synth.potts(K, BETA))
    stream = torch.cuda.Stream()
    reg = m.region_grid(X, 1, B, B, r0, r1, 8, BETA1, stream=stream.cuda_stream)
    del X
    reg.emit_loglik()
    reg.set_labels(np.random.default_rng(SEED).integers(0, K, size=reg.n_window).astype(np.int32))
    ms_sum = time_launches(torch, stream, lambda: reg.posterior_summary(ET), launches)
    ms_estep = time_launches(torch, stream, lambda: reg.estep_stats_async(ET), max(launches // 4, 5))
    n = reg.n
    KP = (K + 7) // 8 * 8
    bytes_node = 8 * KP + 4 + 64 + 28
    gbs = n * bytes_node / (ms_sum * 1e-3) / 1e9
    reg.close()
    m.close()
    return dict(shape=name, n_nodes=n, d=d, K=K, rows=[r0, r1], launches=launches, summary_ms=ms_sum,
                estep_ms=ms_estep, bytes_per_node=bytes_node, achieved_gbs=gbs,
                frac_of_hbm_datasheet=gbs / HBM_DATASHEET_GBS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--shapes", default="cfg5_band,cfg3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the summary kernel is timed on the GPU only")
    import phylo_hmrf_b200 as ph
    from phylo_hmrf_b200 import synth
    res = dict(card=card(), hbm_datasheet_gbs=HBM_DATASHEET_GBS,
               results=[one_shape(torch, ph, synth, s, args.launches) for s in args.shapes.split(",")])
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
