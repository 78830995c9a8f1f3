"""Worker of tests/test_gpu_posterior_summary.py: the one-region problem of tests/em_band_case.py fitted with
posterior_summary=True, in one process or as one rank of a `torchrun` launch (NCCL); writes the gathered
summary."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import em_band_case as case  # noqa: E402


def run(out_dir, B, D, K, m_iter):
    import torch
    from phylo_hmrf_b200.hmrf import phyloHMRF
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as td
        td.init_process_group("nccl", device_id=torch.device("cuda", local))
    X, len_vec, edge_list_vec = case.problem(B, D)
    m = phyloHMRF(n_samples=len(X), n_features=D, observation=X, edge_list_1=edge_list_vec, len_vec=len_vec,
                  n_components=K, estimate_type=case.ET, beta=case.BETA, beta1=case.BETA1, device=local)
    m.init_fn, m.mstep_fn = case.init_fn, case.mstep_fn
    res = m.fit_accumulate_test(X, len_vec, 1e-12, "test", m_iter, n_threads=1, posterior_summary=True)
    np.savez(os.path.join(out_dir, "w%d_rank%d.npz" % (world, rank)), t_labels=res[6],
             n_bands=len(getattr(m, "_bands", {})), **m.posterior_summary_)
    m.close()
    if world > 1:
        td.destroy_process_group()


if __name__ == "__main__":
    run(sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]))
