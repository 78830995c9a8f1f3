"""Command line of the reference (`python phylo_hmrf.py ...`, phylo_hmrf.py:1531-1760) over the
re-hosted model: same option names and code defaults (SURVEY section 5), same cache files, same
`.mat` result.  `--reload 1` reads the `data.*.npy` / `edgelist.*.npy` / `lenvec.*.txt` caches
(phylo_hmrf.py:1676-1690); otherwise the species' Hi-C text files are aligned and preprocessed
(`phylo_hmrf_b200.loader`, image pipeline on the GPU) and the caches are written
(phylo_hmrf.py:1692-1704)."""
from __future__ import annotations

import os
from optparse import OptionParser

import numpy as np


def parse_args(argv=None):
    """phylo_hmrf.py:1531-1568 (33 options; the code defaults, not the README's)."""
    parser = OptionParser(usage="Phylo-HMRF state estimation", add_help_option=False)
    for flags, default in [
        (("-n", "--num_states"), "10"), (("-f", "--chromosome"), "1"), (("-l", "--length"), "one"),
        (("-p", "--root_path"), "."), (("-m", "--multiple"), "true"), (("-a", "--species_name"), "human"),
        (("-o", "--sort_states"), "false"), (("-r", "--run_id"), "0"), (("-c", "--cons_param"), "1"),
        (("-t", "--method_mode"), "1"), (("-d", "--initial_mode"), "0"), (("-i", "--initial_weight"), "0.3"),
        (("-k", "--initial_weight1"), "0.1"), (("-j", "--initial_magnitude"), "1"), (("-s", "--simu_version"), "1"),
        (("-u", "--position1"), "0"), (("-v", "--position2"), "50000"), (("-w", "--filter_sigma"), "0.25"),
        (("-b", "--beta"), "1"), (("--beta1",), "0.5"), (("--num_neighbor",), "8"), (("--filter_mode",), "0"),
        (("-e", "--threshold"), "0.001"), (("-g", "--estimate_type"), "0"), (("-q", "--annotation"), "test"),
        (("--dtype",), "0"), (("--reload",), "0"), (("--quantile",), "1"), (("--miter",), "60"),
        (("--resolution",), "50000"), (("--ref_species",), "hg38"), (("--chromvec",), "1"), (("--output",), "."),
    ]:
        parser.add_option(*flags, default=default)
    opts, _ = parser.parse_args(argv)
    return opts


def _read_table(path, cast):
    with open(path) as f:
        return [[cast(v) for v in line.split('\t')] for line in f if line.strip()]


def _load_raw(opts, data_path, resolution, device):
    """phylo_hmrf.py:1622-1695: species / path lists, chromosome list, the common x_max (median over
    chromosomes and species of the largest contact value), then utility.load_data_chromosome2."""
    from . import loader
    with open("%s/species_name.1.txt" % data_path) as f:
        species = [line.strip() for line in f if line.strip()]
    with open("%s/path_list.txt" % data_path) as f:
        filename_list = [line.strip() for line in f if line.strip()]
    chromvec = str(opts.chromvec)
    chrom_vec = list(range(1, 23)) if chromvec == "-1" else [int(c) for c in chromvec.split(',')]
    ref_filename = "%s/%s.chrom.sizes" % (data_path, str(opts.ref_species))
    qfile = 'chrom_quantile_test.txt'
    if int(opts.quantile) == 0 and os.path.exists(qfile):
        m_values = np.atleast_2d(np.loadtxt(qfile, delimiter='\t'))[:, 6]
    else:
        m_vec_list = loader.quantile_contact_vec(chrom_vec, resolution, ref_filename, filename_list, species)
        np.savetxt(qfile, m_vec_list, fmt='%.4f', delimiter='\t')
        m_values = m_vec_list[:, 6]
    x_max, x_min = float(np.median(m_values)), 0
    return loader.load_data_chromosome2(chrom_vec, x_max, x_min, resolution, int(opts.num_neighbor),
                                        int(opts.filter_mode), float(opts.filter_sigma), int(opts.dtype),
                                        ref_filename, filename_list, species, data_path, str(opts.annotation),
                                        device=device)


def _launch_context(device):
    """(device, rank, world, comm or None).  Under `torchrun` (RANK/LOCAL_RANK/WORLD_SIZE in the
    environment) one process per GPU: the device is LOCAL_RANK, the process binds to the cores next
    to that GPU and joins the NCCL group; files are written by rank 0 only."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return device, 0, 1, None
    import torch
    import torch.distributed as td
    from . import dist as pdist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pdist.bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    if not td.is_initialized():
        td.init_process_group("nccl", device_id=torch.device("cuda", local))
        import atexit
        atexit.register(lambda: td.is_initialized() and td.destroy_process_group())
    return local, td.get_rank(), world, td


def run(opts, device=0):
    """phylo_hmrf.py:1570-1749.  Returns the dict written to the `.mat` file."""
    import scipy.io
    from .hmrf import phyloHMRF
    # the graph cut of every EM iteration: 'host' (csrc/gco.cpp, default) or 'device' (the same swap on the GPU);
    # an environment variable, so that the option list stays the reference's
    graph_cut = os.environ.get("PHMRF_GRAPH_CUT", "host")
    if graph_cut not in ("host", "device"):
        raise SystemExit("PHMRF_GRAPH_CUT must be 'host' or 'device', not %r" % graph_cut)
    device, rank, world, td = _launch_context(device)
    run_id, K = int(opts.run_id), int(opts.num_states)
    cons_param = float(opts.cons_param)
    resolution = int(opts.resolution)
    data_path, output_path = str(opts.root_path), str(opts.output)
    edge_list = _read_table("%s/edge.1.txt" % data_path, int)
    bl = "%s/branch_length.1.txt" % data_path
    branch_list = _read_table(bl, float)[0] if os.path.exists(bl) else None
    stem = "%dKb.observed.%d" % (resolution // 1000, run_id)
    f1, f2, f3 = ("%s/data.%s.npy" % (output_path, stem), "%s/edgelist.%s.npy" % (output_path, stem),
                  "%s/lenvec.%s.txt" % (output_path, stem))
    if int(opts.reload) == 1 and all(os.path.exists(f) for f in (f1, f2, f3)):
        samples = np.load(f1)
        edge_list_vec = list(np.load(f2, allow_pickle=True))
        len_vec = np.atleast_2d(np.loadtxt(f3, dtype='int32', delimiter='\t')).tolist()
    else:   # phylo_hmrf.py:1630-1706: align the species' contact files, build the regions, write the caches
        if rank == 0:
            samples, len_vec, edge_list_vec = _load_raw(opts, data_path, resolution, device)
            os.makedirs(output_path, exist_ok=True)
            np.save(f1, samples)
            ev = np.empty(len(edge_list_vec), dtype=object)
            for i, e in enumerate(edge_list_vec):
                ev[i] = e
            np.save(f2, ev, allow_pickle=True)
            np.savetxt(f3, np.asarray(len_vec), fmt='%d', delimiter='\t')
        if world > 1:       # the other ranks read what rank 0 prepared
            td.barrier()
            if rank != 0:
                samples = np.load(f1)
                edge_list_vec = list(np.load(f2, allow_pickle=True))
                len_vec = np.atleast_2d(np.loadtxt(f3, dtype='int32', delimiter='\t')).tolist()
    if int(opts.method_mode) != 1:
        raise SystemExit("method_mode 1 (Phylo-HMRF) is the only mode of the reference's run()")
    model = phyloHMRF(n_components=K, run_id=run_id, n_samples=samples.shape[0], n_features=samples.shape[-1],
                      observation=samples, edge_list=edge_list, len_vec=len_vec, type_id=int(opts.simu_version),
                      branch_list=branch_list, edge_list_1=edge_list_vec, cons_param=cons_param, beta=float(opts.beta),
                      beta1=float(opts.beta1), initial_mode=int(opts.initial_mode),
                      initial_weight=float(opts.initial_weight), initial_weight1=float(opts.initial_weight1),
                      initial_magnitude=float(opts.initial_magnitude), learning_rate=0.001,
                      estimate_type=int(opts.estimate_type), max_iter=100, n_iter=5000, tol=1e-7, device=device,
                      graph_cut=graph_cut)
    filename = "%s/estimate_ou_%d_%.2f_%d_%s" % (output_path, run_id, cons_param, K, str(opts.annotation))
    res = model.fit_accumulate_test(samples, len_vec, float(opts.threshold), filename, int(opts.miter))
    params_vec1, params_vec2, params_vecList, iter_id1, iter_id2, cost_vec, state_vec = res
    mdict = {'state_vec': state_vec, 'len_vec': np.asarray(len_vec), 'params_vec1': params_vec1,
             'params_vec2': params_vec2, 'iter_id1': iter_id1, 'iter_id2': iter_id2, 'cost_vec': cost_vec}
    if rank == 0:
        os.makedirs(output_path, exist_ok=True)
        scipy.io.savemat("%s/estimate_ou_%d_%.2f_%d.mat" % (output_path, run_id, cons_param, K), mdict)
    model.close()
    return mdict


if __name__ == '__main__':
    run(parse_args())
