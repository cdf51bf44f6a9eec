"""CPU-side checks of the drop-in boundary: libplaidgpu.so loads, exports every symbol that
include/plaidgpu.h declares, refuses to run without a GPU (no CPU fallback), and its host-only
helper (the median combine step of the sharded protocol) matches the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from plaid_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "plaidgpu.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(plaidgpu_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_all_exported_and_typed():
    lib = L.load()
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/plaidgpu.h but not exported"
    assert sorted(L.SYMBOLS) == names, "ctypes table and header disagree"
    assert lib.plaidgpu_version() == 100


def test_struct_layouts_match_header():
    # sizes implied by the header (LP64): matrix 4*4+8+3*8 = 48, opts 8*4+4*8+8+3*8+8 = 104, scalars 5*8+8 = 48
    assert C.sizeof(L.Matrix) == 48
    assert C.sizeof(L.Opts) == 104
    assert C.sizeof(L.Scalars) == 48
    assert L.Scalars.fp64.offset == 44 and L.Scalars.fp64.size == 4
    o = L.Opts()
    L.load().plaidgpu_default_opts(C.byref(o))
    assert (o.scorer, o.stats_mean, o.normalize, o.ignore_zero, o.remove_log2, o.rmax) == (0, 1, 1, -1, -1, 1500.0)


def _no_gpu():
    try:
        import torch
        return not torch.cuda.is_available()
    except Exception:
        return True


@pytest.mark.skipif(not _no_gpu(), reason="only meaningful on a GPU-less box")
def test_no_cpu_fallback():
    lib = L.load()
    h = C.c_void_p()
    assert lib.plaidgpu_init(0, C.byref(h)) == L.ERR_CUDA
    from plaid_b200 import Context
    with pytest.raises(L.PlaidGpuError):
        Context(0)


def test_combine_medians_host_logic():
    from oracle import plaid_oracle as O
    lib = L.load()
    rng = np.random.default_rng(0)
    med_all = rng.normal(size=1000)
    med_nz = rng.normal(size=1000)
    med_all[7] = np.nan  # an all-NaN column: mean(na.rm=TRUE) skips it
    s = L.Scalars()
    assert lib.plaidgpu_combine_medians(-1, 0.0, med_all.ctypes.data, med_nz.ctypes.data, 1000, C.byref(s)) == 0
    assert s.ignore_zero == 1 and s.med_mean == O.r_mean(med_nz)
    assert lib.plaidgpu_combine_medians(-1, -0.5, med_all.ctypes.data, med_nz.ctypes.data, 1000, C.byref(s)) == 0
    assert s.ignore_zero == 0 and s.med_mean == O.r_mean(med_all)
    assert lib.plaidgpu_combine_medians(1, 3.0, med_all.ctypes.data, med_nz.ctypes.data, 1000, C.byref(s)) == 0
    assert s.ignore_zero == 1


def test_rowmap_semantics():
    from plaid_b200 import make_rowmap
    rm = make_rowmap(["a", "b", "a", "c", "zz"], ["c", "a", "q", "a"])
    assert rm.tolist() == [1, -1, -1, 0, -1]  # first occurrence on both sides (R/plaid.R:65-72)


def test_gmt_ingestion_matches_oracle(tmp_path):
    """read.gmt + gmt2mat in C++ behind the ABI (scope row f2) vs the oracle restatement, on the reference's
    bundled hallmarks.gmt and on an adversarial file (comments, CRLF, duplicated set names, NA, blanks)."""
    import ctypes as C
    from oracle.gmt import gmt2mat, read_gmt
    from plaid_b200 import gmt2mat_file
    path = os.path.join(ROOT, "tests", "golden", "hallmarks.gmt")
    got = gmt2mat_file(path)
    D, rn, cn = gmt2mat(read_gmt(path))
    assert got.shape == (4386, 50) == D.shape  # vignette known answer
    assert got.colnames == cn and got.rownames == rn
    assert (got.mat != D).nnz == 0
    tricky = tmp_path / "t.gmt"
    tricky.write_bytes(b"# comment\nS1\tsrc\tA\tB\tNA\tB\t\tC D\r\nS2\tsrc\tB\nS1\tdup\tZ\tY\tX\tW\tV\tU\nS3\tsrc\n"
                       b"S4\tsrc\tA\tQ # trailing comment\tNOTAGENE\nS5\tsrc\tB\tR!second column\tNOTAGENE\n#\n!x\n")
    got = gmt2mat_file(str(tricky))
    D, rn, cn = gmt2mat(read_gmt(str(tricky)))
    assert got.colnames == cn and got.rownames == rn and (got.mat != D).nnz == 0
    assert "NOTAGENE" not in got.rownames and "Q" in got.rownames and "R" in got.rownames  # '#' / '!' cut the line (read.csv)
    # rowmap: first occurrence of a duplicated X rowname wins, unknown names -> -1
    lib = L.load()
    h = C.c_void_p()
    assert lib.plaidgpu_gmt_read(str(tricky).encode(), C.byref(h)) == 0
    last = got.rownames[-1]
    assert last != "B"
    names = [b"B", b"nope", b"B", last.encode()]
    arr = (C.c_char_p * 4)(*names)
    rm = np.empty(4, dtype=np.int32)
    assert lib.plaidgpu_gmt_rowmap(h, arr, 4, rm.ctypes.data) == 0
    assert rm.tolist() == [got.rownames.index("B"), -1, -1, len(got.rownames) - 1]
    lib.plaidgpu_gmt_free(h)
