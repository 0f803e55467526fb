"""ccfindr_b200 -- B200-native variational-Bayes Poisson-NMF engine behind ccfindR's interface.

The compute lives in libvbnmf.so (CUDA, sm_100a; C ABI in include/vbnmf.h).  This package is the
host side: `Engine` (one handle per GPU), the ccfindR-style front ends (`vb_factorize`, `factorize`,
`cluster_id`, `optimal_rank` on `scNMFSet`), the cell / gene QC that precedes them (`filter_cells`,
`filter_genes`, `calc_vmr`, `normalize_count`) and synthetic data generators.
"""
from .api import (calc_vmr, cluster_id, dispersion_from_labels, factorize, filter_cells,
                  filter_genes, normalize_count, optimal_rank, read_10x, remove_zeros, scNMFSet,
                  vb_factorize, write_10x)
from .engine import Comm, Engine

__all__ = ["Engine", "Comm", "scNMFSet", "vb_factorize", "factorize", "cluster_id", "optimal_rank",
           "dispersion_from_labels", "read_10x", "write_10x", "remove_zeros", "filter_cells",
           "filter_genes", "calc_vmr", "normalize_count"]
