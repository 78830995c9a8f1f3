#!/usr/bin/env python
"""bench.py -- node-states/sec per EM iteration (emission + cost arrays + posteriors/costs +
statistics), the metric of BASELINE.json.  GCO and the M-step are excluded by the metric's
definition (SURVEY 8(d)); phase B runs on arg-min labels (the GCO stand-in of 8(d)).

    python bench.py --gpus N --steps K --warmup W           # this repo, one process per GPU
    python bench.py --impl reference --steps K --warmup W   # the reference's CPU path
    python bench.py --workload cfg4_genome_50kb             # another BASELINE configuration
    python bench.py --dump-outputs DIR                      # also write the last timed step's outputs as .npy

A *step* is one pass of the hot path over every region (or row band) this rank holds: phase A1
emission (+max|logp|), A2 integer unary + integer edge weights + per-node maxima, B fused
posteriors/costs/statistics, and for N>1 one NCCL all-reduce of the K(1+d+d^2)+3 statistics.
Every region has its own CUDA stream, so regions overlap (the HBM-bound A2 of one with the
FP64-bound A1/B of another).  Default workload: one row band of the chr1@10kb triangle per GPU
(B=24895 bins, d=9, K=30; weak scaling, at N=8 the bands tile the whole map = config 5).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import queue
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "node-states/sec per EM iteration (emission+costs+stats)"
UNIT = "node-states/s"
BETA, BETA1, ESTIMATE_TYPE = 1.0, 0.1, 3
SEED = 20261017 + 5


def workloads():
    """name -> dict(d, K, regions=[bins of each diagonal region], bands=n or 0, cfg=BASELINE config)"""
    from phylo_hmrf_b200 import synth
    return {
        # BASELINE configs 1 and 2: the shapes of the shipped example (652- and 683-bin synteny
        # regions of chr21/chr22, 4 leaves as shipped); synthetic features here, the shipped
        # files themselves are covered by tests/test_gpu_example_data.py
        "cfg1_chr21_example": dict(d=4, K=10, regions=[652], bands=0, cfg=1),
        "cfg2_chr21_chr22": dict(d=4, K=20, regions=[652, 683], bands=0, cfg=2),
        "cfg3_chr1_50kb": dict(d=5, K=20, regions=[4979], bands=0, cfg=3),
        # 22 autosome regions at 50 kb, 89 321 427 nodes; N>1 deals whole regions to the ranks
        "cfg4_genome_50kb": dict(d=5, K=20, regions=synth.autosome_bins(50000), bands=0, cfg=4),
        # one of the 8 row bands of chr1 at 10 kb per GPU (309 892 960 nodes in all)
        "cfg5_chr1_10kb_band": dict(d=9, K=30, regions=[24895], bands=8, cfg=5),
        "tiny": dict(d=9, K=30, regions=[400], bands=0, cfg=0),
        "mid_d9_k30": dict(d=9, K=30, regions=[5000], bands=0, cfg=0),
    }


def algorithmic_bytes_per_node(d, K):
    return 16 * d + 4 * K + 68  # SURVEY 8(d)


def algorithmic_flops_per_node_state(d):
    return 2 * d * d + 6 * d + 12  # SURVEY 8(d)


def estep_flops_per_node_state(d):
    return 6 + 2 + 2 * d + d * (d + 1)  # posterior arithmetic + packed statistics share of F(d)


def emit_flops_per_node_state(d):
    return d * d + 3 * d + 2


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the
    committed `ncu --set full` capture of this workload (profiles/r2_traffic.json, written by
    tools/ncu_traffic.py from the .ncu-rep); None if the workload was not captured."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        return table[workload][kernel]
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class Piece:
    """One region (or row band) resident on the device, with what the end-to-end leg needs."""

    def __init__(self, m, torch, region_index, B, r0, r1, d, banded, real_gco=False):
        from phylo_hmrf_b200 import synth
        self.B, self.r0, self.r1, self.banded = B, r0, r1, banded
        self.stream = torch.cuda.Stream()
        g = synth.window_xy(B, r0, r1)
        self.n, self.n_window, self.own_offset = g["n_own"], g["n_window"], g["own_offset"]
        # The region is built on the device from the grid geometry (phmrf_region_create_grid): the
        # host only prepares the window's feature rows, no edge array exists on the host.
        X_window = synth.features(SEED + 1000 * region_index, g["x"], g["y"], d)
        g.clear()
        self.reg = m.region_grid(X_window, 1, B, B, r0, r1, 8, BETA1, stream=self.stream.cuda_stream)
        self.E = self.reg.n_edges
        self.X_pin = torch.empty((self.n, d), dtype=torch.float64, pin_memory=True)  # end-to-end leg
        self.X_pin.numpy()[:] = X_window[self.own_offset:self.own_offset + self.n]
        # labels for phase B: arg-min of the integer unary over the *window* (owned + halo rows); the
        # halo labels come from a throw-away region over the window (what the neighbouring bands'
        # graph cuts would have produced)
        if self.n_window != self.n:
            win = m.region(X_window, np.zeros((0, 2), np.int64), np.zeros(0))
            win.emit_loglik()
            win.quantise(want_unary=False, want_edges=False)
            self.labels_window = win.labels_argmin_unary()
            win.close()
        else:
            self.reg.emit_loglik()
            self.reg.quantise(want_unary=False, want_edges=False)
            self.labels_window = self.reg.labels_argmin_unary()
        self.gco_s = None
        if real_gco:        # configs 1-2 (SURVEY 8(d)): the labels of phase B come from the real graph cut, once, untimed
            import phylo_hmrf_b200 as ph
            q = self.reg.quantise(staged=True)
            ids, _ = self.reg.edges()
            t0 = time.perf_counter()
            self.labels_window = ph.gco_cut_int(q["unary_i32"], ids, q["w_i32"], q["V_i32"], n_iter=5000,
                                                algorithm='swap', init_labels=self.labels_window.astype(np.int32))
            self.gco_s = time.perf_counter() - t0
        self.reg.set_labels(self.labels_window)
        self._X_window = X_window      # kept until the end-to-end leg decides whether it needs a twin

    def twin(self, m, torch, d):
        """A second device copy of the same piece on its own stream (end-to-end leg: two batches in
        flight so that one's download overlaps the other's upload)."""
        t = Piece.__new__(Piece)
        t.B, t.r0, t.r1, t.banded = self.B, self.r0, self.r1, self.banded
        t.stream = torch.cuda.Stream()
        X_window = self._X_window
        t.n, t.n_window, t.own_offset = self.n, self.n_window, self.own_offset
        t.reg = m.region_grid(X_window, 1, self.B, self.B, self.r0, self.r1, 8, BETA1, stream=t.stream.cuda_stream)
        t.E = t.reg.n_edges
        t.X_pin = self.X_pin
        t.labels_window = self.labels_window
        t.reg.set_labels(t.labels_window)
        return t


def run_ours(args):
    import torch
    import torch.distributed as dist
    import phylo_hmrf_b200 as ph
    from phylo_hmrf_b200 import synth, engine
    from phylo_hmrf_b200 import dist as pdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    cores = pdist.bind_to_gpu_numa(local_rank)   # before any pinned allocation
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"        # keep NCCL's version banner off stdout: ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    wl = workloads()[args.workload]
    d, K, bins, n_bands = wl["d"], wl["K"], wl["regions"], wl["bands"]
    # model: identical on every rank (a pure function of the seed and the first rows of the first region)
    g0 = synth.make_band(SEED, bins[0], d, 0, min(bins[0], 24), beta1=BETA1)
    means, covars = synth.model(SEED, g0["X_own"], K, d)
    del g0
    V = synth.potts(K, BETA)
    main = torch.cuda.Stream()
    m = ph.Model(K, d, device=local_rank)
    m.set_model(means, covars, V)

    # ---- which pieces this rank holds
    if n_bands:                      # one band of ONE region per GPU (weak scaling)
        r0, r1 = synth.band_rows(bins[0], n_bands)[rank % n_bands]
        specs = [(0, bins[0], r0, r1, True)]
        sharding = "row bands of one region, one per GPU (band %d of %d on rank 0)" % (rank % n_bands, n_bands)
    elif world > 1 and len(bins) >= world:   # whole regions dealt to the ranks by node count
        owner = pdist.assign_regions([b * (b + 1) // 2 for b in bins], world)
        specs = [(i, b, 0, b, False) for i, b in enumerate(bins) if owner[i] == rank]
        sharding = "whole regions dealt to the ranks by node count (dist.assign_regions)"
    else:                            # replicas: every rank runs the whole workload
        specs = [(i, b, 0, b, False) for i, b in enumerate(bins)]
        sharding = "replicas: every rank runs every region" if world > 1 else "single GPU"
    real_gco = wl["cfg"] in (1, 2)
    pieces = [Piece(m, torch, i, b, r0, r1, d, banded, real_gco=real_gco) for (i, b, r0, r1, banded) in specs]
    n_rank = sum(p.n for p in pieces)
    E_rank = sum(p.E for p in pieces)
    stats_len = m.stats_len
    stats_dev = [pdist.stats_tensor(p.reg) for p in pieces]      # the library's device buffers
    absmax_dev = [pdist.absmax_tensor(p.reg) for p in pieces]
    if world > 1 and n_bands:
        pdist.share_weight_max(pieces[0].reg, dist)   # the bands are ONE region: shared down-weight factor
    total_stats = torch.zeros(stats_len, dtype=torch.float64, device="cuda")
    single = len(pieces) == 1

    def enqueue_step(evs=None):
        """One step on every piece's stream; evs[p] = 4 events around the three phases."""
        for pi, p in enumerate(pieces):
            s = p.stream
            if evs is not None:
                evs[pi][0].record(s)
            p.reg.emit_loglik_async()
            if world > 1 and p.banded:           # region-wide max|logp| before the integer conversion
                with torch.cuda.stream(s):
                    dist.all_reduce(absmax_dev[pi], op=dist.ReduceOp.MAX)
            if evs is not None:
                evs[pi][1].record(s)
            p.reg.quantise_async()
            if evs is not None:
                evs[pi][2].record(s)
            p.reg.estep_stats_async(ESTIMATE_TYPE)
            if evs is not None:
                evs[pi][3].record(s)
        if world > 1:
            if single:
                with torch.cuda.stream(pieces[0].stream):
                    dist.all_reduce(stats_dev[0])
            else:                                 # sum over this rank's regions, then across ranks
                done = [torch.cuda.Event() for _ in pieces]
                for pi, p in enumerate(pieces):
                    done[pi].record(p.stream)
                with torch.cuda.stream(main):
                    for e in done:
                        main.wait_event(e)
                    total_stats.zero_()
                    for t in stats_dev:
                        total_stats.add_(t)
                    dist.all_reduce(total_stats)
                    back = torch.cuda.Event()
                    back.record(main)
                for p in pieces:                  # the next step may overwrite the buffers only afterwards
                    p.stream.wait_event(back)

    def fork():
        e = torch.cuda.Event(enable_timing=True)
        e.record(main)
        for p in pieces:
            p.stream.wait_event(e)
        return e

    def join():
        for p in pieces:
            e = torch.cuda.Event()
            e.record(p.stream)
            main.wait_event(e)
        e = torch.cuda.Event(enable_timing=True)
        e.record(main)
        return e

    warm = max(args.warmup, 3)
    for _ in range(warm):
        enqueue_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = engine.launch_count()
    all_evs = []
    t_start = fork()
    for _ in range(args.steps):
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in pieces]
        enqueue_step(evs)
        all_evs.append(evs)
    t_end = join()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = engine.launch_count() - launches0
    total_ms = t_start.elapsed_time(t_end)
    # the last timed step's results, read before the untimed phase-timing steps below run the regions again
    if world > 1 or single:
        final = (stats_dev[0] if single else total_stats).cpu().numpy()
    else:
        final = sum(t_.cpu().numpy() for t_ in stats_dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, final, pieces, K, d)
    phase_ms = np.zeros(3)        # per step, summed over this rank's regions
    if single:
        for evs in all_evs:
            for pe in evs:
                for i in range(3):
                    phase_ms[i] += pe[i].elapsed_time(pe[i + 1])
        phase_ms /= args.steps
        phase_note = "CUDA events around the three phases inside the timed region"
    else:
        # regions overlap on their streams in the timed region, which stretches every per-stream interval;
        # the kernel times come from two extra steps in which the regions run one after the other
        reps = 2
        for _ in range(reps):
            for pi, p in enumerate(pieces):
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                evs[0].record(p.stream)
                p.reg.emit_loglik_async()
                evs[1].record(p.stream)
                p.reg.quantise_async()
                evs[2].record(p.stream)
                p.reg.estep_stats_async(ESTIMATE_TYPE)
                evs[3].record(p.stream)
                p.stream.synchronize()
                for i in range(3):
                    phase_ms[i] += evs[i].elapsed_time(evs[i + 1])
        phase_ms /= reps
        phase_note = ("summed over this rank's regions, each region run alone in two extra steps (in the timed "
                      "region the regions overlap on their own streams)")
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    nodes_total = torch.tensor([float(n_rank)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(nodes_total)
    nodes_total = float(nodes_total.item())
    value = nodes_total * K / (ms_per_step * 1e-3)

    # ---- correctness of what was timed: the posteriors of every node sum to one, so the first K
    # statistics (after the all-reduce) must add up to the number of nodes
    post_sum = float(final[:K].sum())
    expect = nodes_total if world > 1 else float(n_rank)
    if not abs(post_sum - expect) <= 1e-6 * expect:
        raise SystemExit("bench.py: sum of the posterior statistics %.6f != node count %.0f" % (post_sum, expect))

    # ---- end-to-end leg: host buffers in, host results out, every pass; two (or more) batches in
    # flight so that the download of one overlaps the upload and the kernels of the next
    e2e = run_e2e(args, torch, dist, ph, m, pieces, d, K, world, stats_len)

    nodes_f = torch.tensor([float(e2e.pop("_nodes_per_s_local"))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(nodes_f)
    e2e["value"] = float(nodes_f.item()) * K

    if rank != 0:
        for p in pieces:
            p.reg.close()
        m.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (phase B) and of the whole step
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    fp64_peak = engine.probe(0, device=local_rank)  # TFLOP/s, DFMA chains, measured in this run
    F, Bb = algorithmic_flops_per_node_state(d), algorithmic_bytes_per_node(d, K)
    step_s = ms_per_step * 1e-3
    fp64_roof = fp64_peak * 1e12 / F
    hbm_roof = hbm_peak * 1e9 / Bb * K
    bound = "fp64" if fp64_roof < hbm_roof else "hbm"
    b_s = phase_ms[2] * 1e-3
    b_tflops = n_rank * K * estep_flops_per_node_state(d) / b_s / 1e12
    b_bytes = n_rank * (8 * d + 4 + 64)        # SURVEY 8(d): phase B's share of B(d,K)
    if bound == "fp64":
        dominant = {"bound": "fp64", "achieved": b_tflops, "peak": fp64_peak, "unit": "TFLOP/s",
                    "frac": b_tflops / fp64_peak}
    else:
        gbs = b_bytes / b_s / 1e9
        dominant = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak}
    roofline = dict(dominant)
    roofline.update({
        "kernel": "estep_bulk_kernel (phase B: posteriors+costs+statistics, csrc/estep_bulk.cuh)",
        "traffic": ncu_traffic(args.workload, "estep"),
        "peak_source": "FP64: DFMA-chain probe in this run (csrc/probe.cu); HBM: %s" % hbm_src,
        # MEASURED_PEAKS.json has no FP64 figure; the nominal peak (148 SMs x 64 DFMA/clk x 2 x 1.965 GHz) for comparison
        "fp64_peak_nominal": 37.2, "frac_of_nominal_fp64": (b_tflops / 37.2) if bound == "fp64" else None,
        "algorithmic_per_launch": {"flops": n_rank * K * estep_flops_per_node_state(d), "bytes": b_bytes},
        "kernel_share_of_step": phase_ms[2] / phase_ms.sum(),
        "phase_ms": {"A1_emit": phase_ms[0], "A2_quantise": phase_ms[1], "B_estep": phase_ms[2],
                     "note": phase_note},
        "emit_kernel": {"achieved": n_rank * K * emit_flops_per_node_state(d) / (phase_ms[0] * 1e-3) / 1e12,
                        "unit": "TFLOP/s",
                        "frac": n_rank * K * emit_flops_per_node_state(d) / (phase_ms[0] * 1e-3) / 1e12 / fp64_peak},
        "quantise_kernel": {"achieved": (n_rank * K * 12 + E_rank * 12) / (phase_ms[1] * 1e-3) / 1e9, "unit": "GB/s",
                            "frac": (n_rank * K * 12 + E_rank * 12) / (phase_ms[1] * 1e-3) / 1e9 / hbm_peak,
                            "note": "8K read + 4K written per node, 8 read + 4 written per edge"},
        "step": {"node_states_per_s_per_gpu": n_rank * K / step_s, "fp64_roof": fp64_roof, "hbm_roof": hbm_roof,
                 "frac_of_slower_roof": n_rank * K / step_s / min(fp64_roof, hbm_roof),
                 "algorithmic_flops_per_node_state": F, "algorithmic_bytes_per_node": Bb},
    })
    cpu = cpu_vec = None
    if world == 1 and not args.no_cpu:
        cpu = cpu_baseline(d, K, bins[0], seconds=args.cpu_seconds, full_regions=bins if wl["cfg"] in (1, 2) else None)
        cpu_vec = cpu_vectorised(d, K, bins[0])
    resident = sum(p.n * (d * 8 + K * 8 + 96) for p in pieces) / 1e9
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s (BASELINE config %d): %d region(s) of %s bins, d=%d leaves, K=%d states; "
                               "%d nodes on rank 0, %d nodes total"
                               % (args.workload, wl["cfg"], len(bins), bins if len(bins) < 4 else "%d..%d" % (min(bins), max(bins)),
                                  d, K, n_rank, int(nodes_total)),
                   "nodes_per_gpu": n_rank, "edges_per_gpu": E_rank, "estimate_type": ESTIMATE_TYPE, "beta": BETA,
                   "beta1": BETA1,
                   "labels": ("the reference's graph cut itself (GCO alpha-beta swap to convergence on the host, run once "
                              "before the timed region: %.1f s for this rank's regions); GCO and M-step excluded from the metric"
                              % sum(p.gco_s for p in pieces)) if real_gco else
                             "arg-min of the integer unary (GCO stand-in, SURVEY 8(d)); GCO and M-step excluded",
                   "l2": ("inputs per step (X + log-likelihood + graph, %.2f GB) exceed the 126 MB L2; no flush needed"
                          % resident) if resident > 0.3 else
                         ("inputs per step are %.3f GB: they FIT the 126 MB L2 and are not flushed between steps "
                          "(the configuration is this small)" % resident),
                   "parallelism": "%s; all-reduce of %d doubles" % (sharding, stats_len),
                   "cpu_affinity": "cores local to the GPU (NVML), %d cores" % len(cores) if cores else "unchanged",
                   "checked": "sum of the posterior statistics == node count after the all-reduce"},
        "e2e": e2e,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "cpu_vectorised": cpu_vec,
    }
    print(json.dumps(out))
    for p in pieces:
        p.reg.close()
    m.close()
    if world > 1:
        dist.destroy_process_group()


LOGPROB_SAMPLE_ROWS = 65536     # 15.7 MB of float64 at K=30


def dump_outputs(out_dir, final, pieces, K, d):
    """What the last timed step computed, as float64 .npy files for comparing two builds output for output
    (the inputs are a pure function of SEED and the workload):

    * stats_post, stats_obs, stats_obs_obsT, cost_sums: the statistics the step returns (summed over this
      rank's regions and, for N>1, all-reduced) and its three cost sums;
    * logprob_rows: the phase-A1 log-likelihood, a seeded sample of node rows of this rank's pieces
      (logprob_index: piece, node);
    * unary_i32_rows, w_i32, V_i32, dwf: what phase A2 hands to the graph cut -- the integer unary of the
      same nodes, a seeded sample of the integer edge weights (w_index: piece, edge), the integer label
      compatibility and the down-weight factor of each piece.  They are read back with phmrf_quantise,
      which converts the log-likelihood the last step left on the device again; the conversion is exact
      integer arithmetic on the same input, so these are the arrays the step computed."""
    from phylo_hmrf_b200.engine import unpack_stats
    os.makedirs(out_dir, exist_ok=True)
    final = np.asarray(final, dtype=np.float64)
    stats = unpack_stats(final, K, d)
    arrays = {"stats_post": stats["post"], "stats_obs": stats["obs"], "stats_obs_obsT": stats["obs*obs.T"],
              "cost_sums": final[-3:]}
    rng = np.random.default_rng(SEED)
    per_piece = max(1, LOGPROB_SAMPLE_ROWS // len(pieces))
    out = {k: [] for k in ("logprob_rows", "logprob_index", "unary_i32_rows", "w_i32", "w_index", "V_i32", "dwf")}
    for i, p in enumerate(pieces):
        pick = np.sort(rng.choice(p.n, size=min(per_piece, p.n), replace=False))
        lp = p.reg.logprob()
        out["logprob_rows"].append(lp[pick])
        out["logprob_index"].append(np.column_stack([np.full(len(pick), i), pick]))
        del lp
        q = p.reg.quantise(boundary_cap=0)
        out["unary_i32_rows"].append(q["unary_i32"][pick])
        edges = np.sort(rng.choice(p.E, size=min(per_piece, p.E), replace=False))
        out["w_i32"].append(q["w_i32"][edges])
        out["w_index"].append(np.column_stack([np.full(len(edges), i), edges]))
        out["V_i32"].append(q["V_i32"][None])
        out["dwf"].append([q["dwf"]])
        del q
    arrays.update({k: np.concatenate(v) for k, v in out.items()})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_e2e(args, torch, dist, ph, m, pieces, d, K, world, stats_len):
    """End-to-end leg through the C ABI with HOST buffers.  One *pass* = one region: X uploaded
    from pinned memory, emission, integer cost arrays downloaded (the graph cut's inputs), labels
    uploaded (the graph cut's output), E-step, statistics downloaded.  Several passes are in
    flight from worker threads (like the product's thread pool over regions): the copy engines
    work in both directions at once.  For N>1 one all-reduce per step, issued in step order."""
    import ctypes as C
    lib = ph._lib.lib()
    steps = max(1, min(args.steps, args.e2e_steps))
    lanes = list(pieces)
    if len(pieces) == 1 and args.lanes > 1:
        lanes.append(pieces[0].twin(m, torch, d))     # the same band twice: two batches in flight
    for p in pieces:
        p._X_window = None
    device_index = torch.cuda.current_device()
    n_workers = min(len(lanes), max(1, args.lanes if len(pieces) == 1 else args.workers))
    for p in lanes:
        p.unary_pin = ph.engine.pinned_empty((p.n, K), np.int32)
        p.wi_pin = ph.engine.pinned_empty((p.E,), np.int32)
        p.lab_pin = ph.engine.pinned_empty((p.n_window,), np.int32)
        p.lab_pin[:] = p.labels_window
        p.stats_host = np.empty(stats_len - 3)
        p.sums_host = np.empty(3)
        p.V_i32 = np.empty((K, K), np.int32)

    trace = [] if args.e2e_trace else None

    def one_pass(p):
        t = [time.perf_counter()]
        p.reg.update_X(p.X_pin.numpy())                                # H2D: X
        ph._lib.check(lib.phmrf_emit_loglik(p.reg._h, None))
        t.append(time.perf_counter())
        dwf, nb = C.c_double(), C.c_int64()
        ph._lib.check(lib.phmrf_quantise(p.reg._h, 0.0, 1e-9, ph._lib.i32ptr(p.unary_pin), ph._lib.i32ptr(p.wi_pin),
                                         ph._lib.i32ptr(p.V_i32), C.byref(dwf), None, 0, C.byref(nb)))   # D2H: GCO inputs
        t.append(time.perf_counter())
        ph._lib.check(lib.phmrf_set_labels(p.reg._h, ph._lib.i32ptr(p.lab_pin)))    # H2D: labels (GCO output)
        t.append(time.perf_counter())
        ph._lib.check(lib.phmrf_estep_stats(p.reg._h, ESTIMATE_TYPE, None, ph._lib.dptr(p.stats_host),
                                            ph._lib.dptr(p.sums_host)))              # D2H: statistics
        t.append(time.perf_counter())
        if trace is not None:
            trace.append((lanes.index(p), t))

    passes_per_step = len(lanes)
    lock = threading.Lock()
    cond = threading.Condition(lock)
    state = {"done": [0] * (steps + 1), "reduced": 0, "acc": [np.zeros(stats_len) for _ in range(steps + 1)]}
    red_dev = torch.zeros(stats_len, dtype=torch.float64, device="cuda")
    errors = []

    def finish(step, p):
        """Book a finished pass; the pass that completes a step issues that step's all-reduce."""
        with cond:
            state["acc"][step][:stats_len - 3] += p.stats_host
            state["acc"][step][stats_len - 3:] += p.sums_host
            state["done"][step] += 1
            if state["done"][step] < passes_per_step or world == 1:
                return
            while state["reduced"] != step:          # collectives in step order on every rank
                cond.wait()
            red_dev.copy_(torch.from_numpy(state["acc"][step]))
            dist.all_reduce(red_dev)
            torch.cuda.current_stream().synchronize()
            state["reduced"] = step + 1
            cond.notify_all()

    def worker(q):
        torch.cuda.set_device(device_index)      # a new thread starts on device 0
        try:
            while True:
                job = q.get()
                if job is None:
                    return
                step, p = job
                one_pass(p)
                finish(step, p)
        except Exception as exc:  # surfaced after the join
            errors.append(exc)

    def run(n_steps, first_step):
        q = queue.Queue()
        for s in range(n_steps):
            for p in lanes:
                q.put((first_step + s, p))
        for _ in range(n_workers):
            q.put(None)
        ths = [threading.Thread(target=worker, args=(q,)) for _ in range(n_workers)]
        t0 = time.perf_counter()
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    run(1, 0)                                   # warm-up pass over every lane
    if errors:
        raise errors[0]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if trace is not None:
        del trace[:]
    wall = run(steps, 1)
    if errors:
        raise errors[0]
    if trace is not None:
        t00 = min(t[0] for _, t in trace)
        for lane, t in sorted(trace, key=lambda v: v[1][0]):
            sys.stderr.write("e2e lane %d: start %.1f ms | X+emit %.1f | quantise+D2H %.1f | labels %.1f | estep %.1f\n"
                             % (lane, (t[0] - t00) * 1e3, (t[1] - t[0]) * 1e3, (t[2] - t[1]) * 1e3, (t[3] - t[2]) * 1e3,
                                (t[4] - t[3]) * 1e3))
    n_pass_nodes = sum(p.n for p in lanes) * steps
    te = torch.tensor([wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    wall = float(te.item())
    h2d = sum(p.n * d * 8 + p.n_window * 4 for p in lanes)
    d2h = sum(p.n * K * 4 + p.E * 4 + stats_len * 8 for p in lanes)
    twin = len(lanes) != len(pieces)
    return {"_nodes_per_s_local": n_pass_nodes / wall, "unit": UNIT,
            "h2d_bytes_per_step": int(h2d // (2 if twin else 1)), "d2h_bytes_per_step": int(d2h // (2 if twin else 1)),
            "ms_per_step": wall * 1e3 / steps / (2 if twin else 1), "steps": steps * (2 if twin else 1),
            "in_flight": n_workers,
            "how": "public C-ABI calls on host buffers (pinned); %d passes in flight from worker threads, so one "
                   "pass's download overlaps the next one's upload and kernels%s"
                   % (n_workers, "; a step here is one pass over the band (the band is resident twice)" if twin else "")}


# ---------------------------------------------------------------------------------------
# CPU legs (the only place outside tests/ and smoke() that executes oracle/)
# ---------------------------------------------------------------------------------------
def _model_for(d, K, B0):
    from phylo_hmrf_b200 import synth
    g0 = synth.make_band(SEED, B0, d, 0, min(B0, 24), beta1=BETA1)
    return synth.model(SEED, g0["X_own"], K, d)


def _cpu_region(args):
    seed, B, d, K, B0, faithful = args
    from phylo_hmrf_b200 import synth
    from oracle import phmrf_oracle as orc
    try:  # one BLAS/OpenMP thread per region process: the processes already fill the cores
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    g = synth.make_band(seed, B, d, beta1=BETA1)
    means, covars = _model_for(d, K, B0)
    V = synth.potts(K, BETA)
    el = np.column_stack([g["edge_ids"].astype(np.float64), g["edge_dist"]])
    t0 = time.perf_counter()
    orc.estep_region(g["X_own"], means, covars, V, el, BETA1, ESTIMATE_TYPE, faithful=faithful)
    return g["n_own"], time.perf_counter() - t0


def cpu_sample(d, K, B_crop, n_regions, B0, faithful=True):
    """One 'iteration' of the reference's CPU path: one process per region (base.py:357-362),
    each running the loop-faithful restatement of _predict_posteriors minus the graph cut.
    B_crop: bins of every region (int) or one entry per region (list)."""
    import multiprocessing as mp
    sizes = list(B_crop) if isinstance(B_crop, (list, tuple)) else [B_crop] * n_regions
    jobs = [(900 + r, sizes[r], d, K, B0, faithful) for r in range(n_regions)]
    t0 = time.perf_counter()
    if n_regions == 1:
        res = [_cpu_region(jobs[0])]
    else:
        with mp.get_context("fork").Pool(n_regions) as p:
            res = p.map(_cpu_region, jobs)
    wall = time.perf_counter() - t0
    nodes = sum(r[0] for r in res)
    return nodes, wall, max(r[1] for r in res)


def cpu_baseline(d, K, B0, seconds=15.0, full_regions=None):
    if full_regions:      # configs 1-2 are timed IN FULL: every region whole, one process per region (SURVEY 8(d))
        nodes, wall, inner = cpu_sample(d, K, list(full_regions), len(full_regions), B0)
        return {"value": nodes * K / inner, "unit": UNIT, "cores": len(full_regions), "kind": "port",
                "sample": "the whole configuration: %d region(s) of %s bins (%d nodes), d=%d K=%d, one forked process per "
                          "region like base.py:357-362 (the reference's own parallel width); loop-faithful Python-3 "
                          "restatement of phylo_hmrf.py:297-468 (the py2 reference cannot run here); GCO excluded"
                          % (len(full_regions), list(full_regions), nodes, d, K)}
    # configs 3-5: the 2e5-node crop BASELINE.md section 4(5) plans (a 632-bin triangle = 200 028 nodes), one per core --
    # a rate, the path is linear in N.  (The reference itself would give ONE process to a one-region configuration.)
    cores = min(os.cpu_count() or 1, 32)
    B_crop = 632 if seconds >= 10 else 60
    nodes, wall, inner = cpu_sample(d, K, B_crop, cores, B0)
    return {"value": nodes * K / inner, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d regions of a %d-bin triangle (%d nodes each, %d in total), d=%d K=%d, one forked process per "
                      "region like base.py:357-362; loop-faithful Python-3 restatement of phylo_hmrf.py:297-468 "
                      "(the py2 reference cannot run here); GCO excluded; %.1f s of wall time"
                      % (cores, B_crop, nodes // cores, nodes, d, K, wall)}


def cpu_vectorised(d, K, B0):
    """BASELINE.md section 4(2): the same maths as vectorised NumPy (no per-node Python loops), the
    best a CPU does with this formulation; one process, NumPy/BLAS threads as the box gives them."""
    B_crop = 632                       # 200 028 nodes: the 2e5-node crop BASELINE.md section 4(5) plans
    cpu_sample(d, K, 120, 1, B0, faithful=False)    # warm the imports
    nodes, wall, inner = cpu_sample(d, K, B_crop, 1, B0, faithful=False)
    return {"value": nodes * K / inner, "unit": UNIT, "cores": 1, "kind": "port (vectorised NumPy, best-effort CPU)",
            "sample": "one %d-bin triangle (%d nodes), d=%d K=%d, a rate (the path is linear in N); GCO excluded"
                      % (B_crop, nodes, d, K)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workloads()[args.workload]
    d, K, B0 = wl["d"], wl["K"], wl["regions"][0]
    cores = min(os.cpu_count() or 1, 32)
    B_crop = 60
    for _ in range(min(args.warmup, 1)):
        cpu_sample(d, K, B_crop, cores, B0)
    tot_nodes, tot_t = 0, 0.0
    for _ in range(args.steps):
        nodes, wall, inner = cpu_sample(d, K, B_crop, cores, B0)
        tot_nodes += nodes
        tot_t += inner
    value = tot_nodes * K / tot_t
    sample = ("each step = %d regions of a %d-bin triangle (%d nodes), d=%d K=%d, one forked process per region "
              "(the reference's own parallel width, base.py:357-362); loop-faithful Python-3 port of "
              "phylo_hmrf.py:297-468 because the py2 reference cannot be imported; GCO excluded like the GPU arm"
              % (cores, B_crop, tot_nodes // args.steps, d, K))
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_t / args.steps * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "%s (bounded sample: %s)" % (args.workload, sample)},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5_chr1_10kb_band", choices=sorted(workloads()))
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--lanes", type=int, default=2, help="end-to-end leg: batches in flight for a one-region workload")
    ap.add_argument("--workers", type=int, default=4, help="end-to-end leg: worker threads over the regions")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-trace", action="store_true", help="per-call wall times of the end-to-end passes on stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
