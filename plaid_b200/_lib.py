"""ctypes binding of libplaidgpu.so (the C ABI in include/plaidgpu.h).

This is the same binding surface the R `.Call` shim uses (rpkg/src/shim.c); Python is only
the host language of the tests / bench in this repository.  Loading fails loudly when the
library has not been built (`python -c "import __graft_entry__ as g; g.build()"` or
`make -C plaid_b200/csrc`); there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

HOST, DEVICE = 0, 1
CSC, DENSE = 0, 1
PLAID, SCSE, SING, SSGSEA, UCELL, AUCELL, GSVA = range(7)
TIES = {"average": 0, "min": 1, "max": 2, "first": 3, "last": 4, "dense": 5}
ROWTF_Z, ROWTF_ECDF, ROWTF_DONE = 0, 1, 2
FILE_RAW, FILE_NPY = 0, 1

OK, ERR_ARG, ERR_CUDA, ERR_NOOVERLAP, ERR_STATE, ERR_NOMEM = 0, -1, -2, -3, -4, -5

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libplaidgpu.so")


class Matrix(C.Structure):
    _fields_ = [("kind", C.c_int32), ("location", C.c_int32), ("P", C.c_int32), ("_pad", C.c_int32),
                ("N", C.c_int64), ("p", C.c_void_p), ("i", C.c_void_p), ("x", C.c_void_p)]


class Opts(C.Structure):
    _fields_ = [("scorer", C.c_int32), ("stats_mean", C.c_int32), ("normalize", C.c_int32),
                ("ignore_zero", C.c_int32), ("remove_log2", C.c_int32), ("score_mean", C.c_int32),
                ("out_location", C.c_int32), ("tile_sets", C.c_int32), ("alpha", C.c_double),
                ("rmax", C.c_double), ("auc_max_rank", C.c_double), ("tau", C.c_double),
                ("nrow_x", C.c_int64), ("matg_full_colsums", C.c_void_p), ("row_mean", C.c_void_p),
                ("row_sd", C.c_void_p), ("gsva_ecdf", C.c_int32), ("exact_fp64", C.c_int32)]


class Scalars(C.Structure):
    _fields_ = [("x_min", C.c_double), ("x_max", C.c_double), ("rank_max", C.c_double),
                ("score_min", C.c_double), ("med_mean", C.c_double), ("ignore_zero", C.c_int32),
                ("_pad", C.c_int32)]


# every symbol include/plaidgpu.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "plaidgpu_init": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "plaidgpu_destroy": (None, [C.c_void_p]),
    "plaidgpu_last_error": (C.c_char_p, [C.c_void_p]),
    "plaidgpu_version": (C.c_int, []),
    "plaidgpu_default_opts": (None, [C.POINTER(Opts)]),
    "plaidgpu_set_genesets": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "plaidgpu_score": (C.c_int, [C.c_void_p, C.POINTER(Matrix), C.c_void_p, C.POINTER(Opts), C.c_void_p]),
    "plaidgpu_score_begin": (C.c_int, [C.c_void_p, C.POINTER(Matrix), C.c_void_p, C.POINTER(Opts), C.POINTER(Scalars)]),
    "plaidgpu_score_compute": (C.c_int, [C.c_void_p, C.POINTER(Scalars), C.c_void_p]),
    "plaidgpu_get_col_medians": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "plaidgpu_get_col_medians_for": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "plaidgpu_combine_medians": (C.c_int, [C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Scalars)]),
    "plaidgpu_score_finish": (C.c_int, [C.c_void_p, C.POINTER(Scalars), C.c_void_p]),
    "plaidgpu_crossprod": (C.c_int, [C.c_void_p, C.POINTER(Matrix), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "plaidgpu_row_moments": (C.c_int, [C.c_void_p, C.POINTER(Matrix), C.c_void_p, C.c_void_p]),
    "plaidgpu_row_ecdf": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int]),
    "plaidgpu_colranks": (C.c_int, [C.c_void_p, C.POINTER(Matrix), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "plaidgpu_group_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int, C.c_void_p]),
    "plaidgpu_group_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "plaidgpu_design_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int, C.c_int,
                                        C.c_void_p]),
    "plaidgpu_score_design_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                              C.c_void_p]),
    "plaidgpu_score_design_stats_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                    C.c_void_p, C.c_int, C.c_void_p]),
    "plaidgpu_col_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p]),
    "plaidgpu_normalize_medians": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "plaidgpu_gmt_read": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "plaidgpu_gmt_from_buffer": (C.c_int, [C.c_char_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "plaidgpu_gmt_free": (None, [C.c_void_p]),
    "plaidgpu_gmt_num_sets": (C.c_int64, [C.c_void_p]),
    "plaidgpu_gmt_num_genes": (C.c_int64, [C.c_void_p]),
    "plaidgpu_gmt_nnz": (C.c_int64, [C.c_void_p]),
    "plaidgpu_gmt_set_name": (C.c_char_p, [C.c_void_p, C.c_int64]),
    "plaidgpu_gmt_gene_name": (C.c_char_p, [C.c_void_p, C.c_int64]),
    "plaidgpu_gmt_csc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "plaidgpu_gmt_rowmap": (C.c_int, [C.c_void_p, C.POINTER(C.c_char_p), C.c_int32, C.c_void_p]),
    "plaidgpu_score_to_file": (C.c_int, [C.c_void_p, C.POINTER(Matrix), C.c_void_p, C.POINTER(Opts), C.c_char_p, C.c_int]),
    "plaidgpu_spmat_read_rda": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    "plaidgpu_spmat_read_mtx": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "plaidgpu_spmat_read_10x": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "plaidgpu_spmat_free": (None, [C.c_void_p]),
    "plaidgpu_spmat_view": (C.c_int, [C.c_void_p, C.POINTER(Matrix)]),
    "plaidgpu_spmat_nnz": (C.c_int64, [C.c_void_p]),
    "plaidgpu_spmat_num_rownames": (C.c_int64, [C.c_void_p]),
    "plaidgpu_spmat_num_colnames": (C.c_int64, [C.c_void_p]),
    "plaidgpu_spmat_rowname": (C.c_char_p, [C.c_void_p, C.c_int64]),
    "plaidgpu_spmat_colname": (C.c_char_p, [C.c_void_p, C.c_int64]),
    "plaidgpu_io_error": (C.c_char_p, []),
    "plaidgpu_launch_count": (C.c_int64, [C.c_void_p]),
    "plaidgpu_reset_launch_count": (None, [C.c_void_p]),
    "plaidgpu_last_kernel_ms": (C.c_double, [C.c_void_p, C.c_int]),
    "plaidgpu_stream": (C.c_void_p, [C.c_void_p]),
    "plaidgpu_plan_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64),
                                     C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32)]),
    "plaidgpu_score_group_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "plaidgpu_score_group_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "plaidgpu_score_group_stats_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_int, C.c_void_p]),
    "plaidgpu_score_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p]),
    "plaidgpu_score_topk_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                             C.c_int, C.c_void_p, C.c_void_p]),
    "plaidgpu_score_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "plaidgpu_tc_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "plaidgpu_tail_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
}

_lib = None


class PlaidGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libplaidgpu error {code}: {msg}")
        self.code = code
        self.msg = msg


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load libplaidgpu.so and type every entry point.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            f"{_LIB_PATH} not found: build it with `make -C plaid_b200/csrc` "
            "(or __graft_entry__.build()). plaid_b200 has no CPU fallback.")
    lib = C.CDLL(os.environ.get("PLAIDGPU_LIB", _LIB_PATH))  # PLAIDGPU_LIB: development builds only
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
