"""phylo_hmrf_b200 -- B200-native (sm_100a) implementation of Phylo-HMRF's per-iteration
E-step hot path behind the reference's own method signatures.  See DESIGN.md."""
from .engine import (Model, Region, PhmrfError, costs_from_sums, cut_general_graph, gco_cut_int, gco_swap_device,
                     log_multivariate_normal_density, unpack_stats)
from .hmrf import phyloHMRF

__all__ = ["Model", "Region", "PhmrfError", "phyloHMRF", "cut_general_graph", "gco_cut_int", "gco_swap_device",
           "log_multivariate_normal_density", "costs_from_sums", "unpack_stats"]
