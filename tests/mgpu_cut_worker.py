"""Worker of tests/test_gpu_graph_cut.py: one rank of a two-rank `torchrun` run of the real `phyloHMRF` on the
banded region of tests/em_band_case.py, with the graph cut on the host or on the device."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import em_band_case as case  # noqa: E402

B, D, K, M_ITER = 96, 5, 8, 8


def run(out_dir, graph_cut):
    import torch
    import torch.distributed as td
    from phylo_hmrf_b200.hmrf import phyloHMRF
    local = int(os.environ["LOCAL_RANK"])
    rank = int(os.environ["RANK"])
    torch.cuda.set_device(local)
    td.init_process_group("nccl", device_id=torch.device("cuda", local))
    X, len_vec, edge_list_vec = case.problem(B, D)
    m = phyloHMRF(n_samples=len(X), n_features=D, observation=X, edge_list_1=edge_list_vec, len_vec=len_vec,
                  n_components=K, estimate_type=case.ET, beta=case.BETA, beta1=case.BETA1, device=local,
                  graph_cut=graph_cut)
    m.init_fn, m.mstep_fn = case.init_fn, case.mstep_fn
    res = m.fit_accumulate_test(X, len_vec, 1e-12, "test", M_ITER, n_threads=1)
    np.savez(os.path.join(out_dir, "%s_rank%d.npz" % (graph_cut, rank)), cost_vec=res[5], t_labels=res[6],
             labels_local=m.labels_local, n_bands=len(getattr(m, "_bands", {})))
    m.close()
    td.destroy_process_group()


if __name__ == "__main__":
    run(sys.argv[1], sys.argv[2])
