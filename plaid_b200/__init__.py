"""plaid_b200 — B200-native implementation of the bigomics/plaid gene-set scoring hot path.

The numeric work is libplaidgpu.so (hand-written sm_100a CUDA, C ABI in include/plaidgpu.h);
this package is the host-side mirror of the reference's R interface used by tests and bench.
Importing the package does not need a GPU; calling any scorer does (no CPU fallback).
"""
from .api import (Context, DeviceCSC, DeviceDense, NamedMatrix, chunked_crossprod, col_topk, colranks, default_context,
                  design_qr, design_stats, gmt2mat_file, group_moments, group_stats, lm_from_moments, make_rowmap,
                  normalize_medians, plaid, plaid_lm, plaid_test, plaid_test_groups, replaid_aucell, replaid_gsva, replaid_scse,
                  replaid_sing, replaid_ssgsea, replaid_ucell, sparse_colranks, read_rda, read_mtx, read_10x, score_to_file,
                  score_design_stats, score_group_moments, score_group_stats, score_topk)

__all__ = ["Context", "DeviceCSC", "DeviceDense", "NamedMatrix", "chunked_crossprod", "col_topk", "colranks",
           "default_context", "design_qr", "design_stats", "gmt2mat_file", "group_moments", "group_stats",
           "lm_from_moments", "make_rowmap", "normalize_medians", "plaid", "plaid_lm", "plaid_test",
           "plaid_test_groups", "replaid_aucell", "replaid_gsva", "replaid_scse",
           "replaid_sing", "replaid_ssgsea", "replaid_ucell", "sparse_colranks", "read_rda", "read_mtx", "read_10x",
           "score_to_file", "score_design_stats", "score_group_moments", "score_group_stats", "score_topk"]
