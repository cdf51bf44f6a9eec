"""Host-side mirror of the reference's R interface for the gene-set scoring hot path.

Same function names, argument meaning, defaults and error behaviour as the exported R
functions (reference `R/plaid.R`, `NAMESPACE:3-16`), so the parity tests read like tests of
the R package:

    plaid(X, matG, stats="mean", chunk=None, normalize=True)        R/plaid.R:60-87
    chunked_crossprod(x, y, chunk=None)                              R/plaid.R:100-123
    normalize_medians(x, ignore_zero=None)                           R/plaid.R:554-575
    colranks(X, sparse=None, signed=False, keep_zero=False, ties_method="average")  :589-623
    sparse_colranks(X, signed=False, ties_method="average")          R/plaid.R:631-650
    replaid_scse / replaid_sing / replaid_ssgsea / replaid_ucell / replaid_aucell   :155-309

Everything numeric happens in libplaidgpu.so (hand-written sm_100a CUDA) through the C ABI
of include/plaidgpu.h.  What stays on the host is exactly what stays in R in the drop-in
package (rpkg/R/plaid.R): matching rows by NAME (intersect/match) and dimnames.  There is
no CPU fallback: without the library or without a B200 these functions raise.

Matrices: `NamedMatrix(mat, rownames, colnames)`; `mat` is a scipy.sparse matrix (R
dgCMatrix), a 2-D numpy array (R base matrix) or a `DeviceCSC` / CUDA torch tensor for
device-resident pipelines.
"""
from __future__ import annotations

import ctypes as C
import math
import sys
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _lib as L

try:  # scipy is only needed to recognise / build sparse inputs
    import scipy.sparse as sp
except Exception:  # pragma: no cover
    sp = None


@dataclass
class NamedMatrix:
    mat: object
    rownames: Optional[Sequence[str]] = None
    colnames: Optional[Sequence[str]] = None

    @property
    def shape(self):
        return tuple(self.mat.shape)


@dataclass
class DeviceCSC:
    """A dgCMatrix whose slots are CUDA torch tensors (p int32[N+1], i int32[nnz], x float64[nnz])."""
    p: object
    i: object
    x: object
    shape: tuple

    @property
    def nnz(self):
        return int(self.x.numel())


def _message(msg: str):  # R message(): stderr
    print(msg, file=sys.stderr)


# ---------------------------------------------------------------------------------------
# context handling
# ---------------------------------------------------------------------------------------
class Context:
    """One libplaidgpu context = one GPU (`plaidgpu_init`)."""

    def __init__(self, device: int = 0):
        self.lib = L.load()
        h = C.c_void_p()
        rc = self.lib.plaidgpu_init(int(device), C.byref(h))
        if rc != L.OK:
            raise L.PlaidGpuError(rc, f"plaidgpu_init(device={device}) failed: no usable sm_100 GPU "
                                      "(plaid_b200 has no CPU fallback)")
        self.h = h
        self.device = device
        self._keep = []  # host arrays that must outlive a call
        self._gkey = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.plaidgpu_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int):
        if rc != L.OK:
            raise L.PlaidGpuError(rc, (self.lib.plaidgpu_last_error(self.h) or b"").decode())

    # -- gene sets -------------------------------------------------------------------------
    def set_genesets(self, G):
        """Register matG (genes x sets, scipy sparse).  Values only matter as zero / non-zero."""
        if G is getattr(self, "_glast", None):  # same object as last time: nothing to do (the caller must
            return                               # not mutate a registered matrix in place)
        G0 = G
        G = sp.csc_matrix(G)
        if G.nnz >= 2 ** 31 or G.shape[0] >= 2 ** 31:
            raise ValueError("matG has 2^31 or more stored entries / rows (dgCMatrix slots are int32)")
        if not G.has_sorted_indices:
            G = G.copy()  # never reorder the caller's arrays
            G.sort_indices()
        key = (G.shape, G.nnz, hash(G.indptr.tobytes()), hash(G.indices.tobytes()), hash(G.data.tobytes()))
        if key == self._gkey:
            self._glast = G0
            return
        gp = np.ascontiguousarray(G.indptr, dtype=np.int32)
        gi = np.ascontiguousarray(G.indices, dtype=np.int32)
        gx = np.ascontiguousarray(G.data, dtype=np.float64)
        self.check(self.lib.plaidgpu_set_genesets(self.h, G.shape[0], G.shape[1], gp.ctypes.data,
                                                  gi.ctypes.data, gx.ctypes.data))
        self._gkey = key
        self._glast = G0  # only after the C call succeeded: a failed registration is retried
        self.n_sets = int(G.shape[1])

    def launch_count(self) -> int:
        return int(self.lib.plaidgpu_launch_count(self.h))

    def kernel_ms(self, which: int) -> float:
        return float(self.lib.plaidgpu_last_kernel_ms(self.h, which))

    def plan_info(self) -> dict:
        ts, nt, wp, ct, gk, gb = (C.c_int32() for _ in range(6))
        nm = C.c_int64()
        self.check(self.lib.plaidgpu_plan_info(self.h, C.byref(ts), C.byref(nt), C.byref(nm), C.byref(wp), C.byref(ct),
                                               C.byref(gk), C.byref(gb)))
        tr, tp, tsl = (C.c_int32() for _ in range(3))
        self.check(self.lib.plaidgpu_tc_info(self.h, C.byref(tr), C.byref(tp), C.byref(tsl)))
        tlr, tlc = C.c_int32(), C.c_int32()
        self.check(self.lib.plaidgpu_tail_info(self.h, C.byref(tlr), C.byref(tlc)))
        return {"tile_sets": ts.value, "n_tiles": nt.value, "nnz_mapped": nm.value, "warps_per_cta": wp.value,
                "ctas": ct.value, "gather_block": gk.value, "gather_blocks": gb.value,
                "tc_rows": tr.value, "tc_rows_padded": tp.value, "tc_slices": tsl.value,
                "tail_rows": tlr.value, "tail_tile_cells": tlc.value}


_default_ctx: dict = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


# ---------------------------------------------------------------------------------------
# marshalling
# ---------------------------------------------------------------------------------------
def _is_torch(t) -> bool:
    return type(t).__module__.startswith("torch")


def _ptr(a):
    if a is None:
        return None
    if _is_torch(a):
        return a.data_ptr()
    return a.ctypes.data


def _matrix_struct(m, keep: list) -> L.Matrix:
    """Describe X for the C ABI.  `keep` receives the arrays that back the pointers."""
    M = L.Matrix()
    if isinstance(m, DeviceCSC):
        M.kind, M.location = L.CSC, L.DEVICE
        M.P, M.N = int(m.shape[0]), int(m.shape[1])
        M.p, M.i, M.x = m.p.data_ptr(), m.i.data_ptr(), m.x.data_ptr()
        keep.append(m)
        return M
    if _is_torch(m):
        if m.dim() != 2:
            raise ValueError("dense device X must be 2-D")
        # R layout is column-major: a torch tensor of shape (N, P) contiguous == P x N column-major
        raise TypeError("pass dense device matrices as DeviceDense(t_colmajor, shape)")
    if isinstance(m, DeviceDense):
        M.kind, M.location = L.DENSE, L.DEVICE
        M.P, M.N = int(m.shape[0]), int(m.shape[1])
        M.x = m.x.data_ptr()
        keep.append(m)
        return M
    if sp is not None and sp.issparse(m):
        m = sp.csc_matrix(m)
        if m.nnz >= 2 ** 31 or m.shape[0] >= 2 ** 31:  # dgCMatrix slots are int32; scipy switches to int64 silently
            raise ValueError("X has 2^31 or more stored entries / rows: split the columns into shards (plaid_b200.sharded)")
        if not m.has_sorted_indices:
            m = m.copy()  # csc_matrix(m) shares buffers with a CSC input: never reorder the caller's arrays
            m.sort_indices()
        p = np.ascontiguousarray(m.indptr, dtype=np.int32)
        i = np.ascontiguousarray(m.indices, dtype=np.int32)
        x = np.ascontiguousarray(m.data, dtype=np.float64)
        keep += [p, i, x]
        M.kind, M.location = L.CSC, L.HOST
        M.P, M.N = int(m.shape[0]), int(m.shape[1])
        M.p, M.i, M.x = p.ctypes.data, i.ctypes.data, x.ctypes.data
        return M
    a = np.asarray(m, dtype=np.float64)
    if a.ndim == 1:  # a bare vector is one sample (R/plaid.R:63)
        a = a[:, None]
    a = np.asfortranarray(a)
    keep.append(a)
    M.kind, M.location = L.DENSE, L.HOST
    M.P, M.N = int(a.shape[0]), int(a.shape[1])
    M.x = a.ctypes.data
    return M


@dataclass
class DeviceDense:
    """Column-major P x N float64 matrix in device memory (a 1-D or (N, P)-contiguous CUDA tensor)."""
    x: object
    shape: tuple


def make_rowmap(x_rownames: Sequence[str], g_rownames: Sequence[str]) -> np.ndarray:
    """rowmap[r] = row of matG aligned with X row r, or -1: `intersect(rownames(X), rownames(matG))`
    + `X[gg,]` / `matG[gg,]` (R/plaid.R:65-72) — first occurrence of a duplicated name wins."""
    gpos = {}
    for k, n in enumerate(g_rownames):
        gpos.setdefault(n, k)
    out = np.full(len(x_rownames), -1, dtype=np.int32)
    seen = set()
    for r, n in enumerate(x_rownames):
        if n in seen:
            continue
        seen.add(n)
        k = gpos.get(n)
        if k is not None:
            out[r] = k
    return out


# every add in fp64 (plaidgpu_opts.exact_fp64) instead of the tensor-core fixed-point block pass; module-wide
# default of the Python mirror, overridable per call through opts_kw
EXACT_FP64 = False


def _opts(lib, **kw) -> L.Opts:
    o = L.Opts()
    lib.plaidgpu_default_opts(C.byref(o))
    o.exact_fp64 = 1 if EXACT_FP64 else 0
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def _score(X: NamedMatrix, matG: NamedMatrix, opts_kw: dict, ctx, out=None):
    """`ctx`: a Context, None (default context of device 0) or a list of Contexts on different devices — the
    columns are then sharded over them by plaidgpu_score_multi (host buffers only)."""
    ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else None
    ctx = (ctxs[0] if ctxs else ctx) or default_context()
    Xm = X.mat
    xr = X.rownames
    if xr is None or matG.rownames is None:
        _message("[plaid] ERROR. No overlapping features.")  # NULL rownames: intersect() is empty
        return None
    rowmap = make_rowmap(xr, matG.rownames)
    if not (rowmap >= 0).any():  # R/plaid.R:66-69
        _message("[plaid] ERROR. No overlapping features.")
        return None
    for cx in (ctxs or [ctx]):
        cx.set_genesets(matG.mat)
    keep: list = []
    M = _matrix_struct(Xm, keep)
    if M.P != len(xr):
        raise ValueError("rownames(X) does not match nrow(X)")
    S = int(matG.mat.shape[1])
    if out is None:
        res = np.empty((S, M.N), dtype=np.float64, order="F")
        out_loc, out_ptr = L.HOST, res.ctypes.data
    else:  # caller-provided buffer: numpy F-order or CUDA tensor holding S x N column-major
        res = out
        out_loc = L.DEVICE if (_is_torch(out) and out.is_cuda) else L.HOST
        out_ptr = _ptr(out)
    o = _opts(ctx.lib, out_location=out_loc, **opts_kw)
    if ctxs and len(ctxs) > 1:
        hs = (C.c_void_p * len(ctxs))(*[cx.h for cx in ctxs])
        rc = ctx.lib.plaidgpu_score_multi(hs, len(ctxs), C.byref(M), rowmap.ctypes.data, C.byref(o), out_ptr)
    else:
        rc = ctx.lib.plaidgpu_score(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), out_ptr)
    if rc == L.ERR_NOOVERLAP:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.check(rc)
    return NamedMatrix(res, list(matG.colnames) if matG.colnames is not None else None,
                       list(X.colnames) if X.colnames is not None else None)


# ---------------------------------------------------------------------------------------
# the reference's functions
# ---------------------------------------------------------------------------------------
def plaid(X: NamedMatrix, matG: NamedMatrix, stats="mean", chunk=None, normalize=True, *, ctx=None, out=None):
    """`plaid(X, matG, stats=c("mean","sum"), chunk=NULL, normalize=TRUE)` (R/plaid.R:60-87).
    `chunk` is accepted and ignored, as in the reference (its value never reaches
    chunked_crossprod, R/plaid.R:80).  Returns NamedMatrix(S x N) or None on no overlap."""
    if isinstance(stats, (list, tuple)):
        stats = stats[0]
    return _score(X, matG, dict(scorer=L.PLAID, stats_mean=1 if stats == "mean" else 0,
                                normalize=1 if normalize else 0), ctx, out)


def chunked_crossprod(x, y, chunk=None, *, ctx=None):
    """`chunked_crossprod(x, y, chunk=NULL)` (R/plaid.R:100-123): t(x) %*% y for a sparse x whose
    non-zeros are constant within a column (the only form plaid() ever passes: G or
    colScale(G, 1/sumG)).  Returns a dense S x N array (documented deviation: the reference
    returns a Matrix-class object on its un-chunked branch).  The chunk message of the
    reference is kept; device-side the product is tiled by columns independently of `chunk`."""
    ctx = ctx or default_context()
    xs = sp.csc_matrix(x)
    xs.sort_indices()
    S = xs.shape[1]
    scale = np.ones(S)
    d = xs.data
    for s in range(S):
        seg = d[xs.indptr[s]:xs.indptr[s + 1]]
        seg = seg[seg != 0]
        if seg.size:
            if not np.all(seg == seg[0]):
                raise ValueError("chunked_crossprod: x must be column-scaled binary (as plaid() builds it)")
            scale[s] = seg[0]
    if chunk is None or chunk < 0:
        chunk = int(round(0.8 * 2147483647 / S))
    ncol_y = y.shape[1] if getattr(y, "ndim", 2) == 2 else 1
    if ncol_y >= chunk:
        _message(f"[chunked_crossprod] chunked compute: chunk = {chunk}")
    ctx.set_genesets(xs)
    keep: list = []
    M = _matrix_struct(y, keep)
    if M.P != xs.shape[0]:
        raise ValueError("non-conformable arguments")
    rowmap = np.arange(M.P, dtype=np.int32)
    res = np.empty((S, M.N), dtype=np.float64, order="F")
    ctx.check(ctx.lib.plaidgpu_crossprod(ctx.h, C.byref(M), rowmap.ctypes.data, scale.ctypes.data, L.HOST,
                                         res.ctypes.data))
    return res


def normalize_medians(x, ignore_zero: Optional[bool] = None, *, ctx=None):
    """`normalize_medians(x, ignore.zero=NULL)` (R/plaid.R:554-575)."""
    ctx = ctx or default_context()
    a = np.asfortranarray(np.asarray(x, dtype=np.float64))
    if a.ndim == 1:
        a = np.asfortranarray(a[:, None])
    res = np.empty_like(a, order="F")
    iz = -1 if ignore_zero is None else int(bool(ignore_zero))
    ctx.check(ctx.lib.plaidgpu_normalize_medians(ctx.h, a.ctypes.data, a.shape[0], a.shape[1], iz, L.HOST,
                                                 res.ctypes.data))
    return res


def sparse_colranks(X, signed: bool = False, ties_method: str = "average", *, ctx=None):
    """`sparse_colranks(X, signed, ties.method)` (R/plaid.R:631-650): csc_matrix, same pattern."""
    ctx = ctx or default_context()
    if ties_method not in L.TIES or ties_method == "dense":  # base::rank has no "dense"; "random" draws from R's RNG
        raise ValueError(f"ties.method {ties_method!r} not supported (average, min, max, first, last)")
    m = sp.csc_matrix(X).astype(np.float64)
    m.sort_indices()
    keep: list = []
    M = _matrix_struct(m, keep)
    r = np.empty(m.nnz, dtype=np.float64)
    ctx.check(ctx.lib.plaidgpu_colranks(ctx.h, C.byref(M), L.TIES[ties_method], int(signed), 1, L.HOST,
                                        r.ctypes.data))
    return sp.csc_matrix((r, m.indices.copy(), m.indptr.copy()), shape=m.shape)


def colranks(X, sparse: Optional[bool] = None, signed: bool = False, keep_zero: bool = False,
             ties_method: str = "average", *, ctx=None):
    """`colranks(X, sparse=NULL, signed=FALSE, keep.zero=FALSE, ties.method="average")`
    (R/plaid.R:589-623).  csc_matrix for (sparse & keep_zero), else a dense P x N array."""
    ctx = ctx or default_context()
    if ties_method not in L.TIES:
        raise ValueError(f"ties.method {ties_method!r} not supported (average, min, max, first, last, dense)")
    is_sp = sp is not None and sp.issparse(X)
    if sparse is None:
        sparse = is_sp
    if sparse and keep_zero:
        return sparse_colranks(X, signed=signed, ties_method=ties_method, ctx=ctx)
    keep: list = []
    if sparse:
        M = _matrix_struct(sp.csc_matrix(X), keep)
    else:
        M = _matrix_struct(X.toarray() if is_sp else X, keep)
    res = np.empty((M.P, M.N), dtype=np.float64, order="F")
    ctx.check(ctx.lib.plaidgpu_colranks(ctx.h, C.byref(M), L.TIES[ties_method], int(signed), 0, L.HOST,
                                        res.ctypes.data))
    return res


def replaid_scse(X: NamedMatrix, matG: NamedMatrix, removeLog2: Optional[bool] = None, scoreMean: bool = False,
                 *, ctx=None, out=None):
    """`replaid.scse(X, matG, removeLog2=NULL, scoreMean=FALSE)` (R/plaid.R:155-190)."""
    rl = -1 if removeLog2 is None else int(bool(removeLog2))
    return _score(X, matG, dict(scorer=L.SCSE, remove_log2=rl, score_mean=int(bool(scoreMean))), ctx, out)


def replaid_sing(X: NamedMatrix, matG: NamedMatrix, *, ctx=None, out=None):
    """`replaid.sing(X, matG)` (R/plaid.R:213-219)."""
    return _score(X, matG, dict(scorer=L.SING, nrow_x=int(X.shape[0])), ctx, out)


def replaid_ssgsea(X: NamedMatrix, matG: NamedMatrix, alpha: float = 0.0, *, ctx=None, out=None):
    """`replaid.ssgsea(X, matG, alpha=0)` (R/plaid.R:244-255)."""
    return _score(X, matG, dict(scorer=L.SSGSEA, alpha=float(alpha)), ctx, out)


def replaid_ucell(X: NamedMatrix, matG: NamedMatrix, rmax: float = 1500, *, ctx=None, out=None):
    """`replaid.ucell(X, matG, rmax=1500)` (R/plaid.R:276-282)."""
    return _score(X, matG, dict(scorer=L.UCELL, rmax=float(rmax)), ctx, out)


def replaid_aucell(X: NamedMatrix, matG: NamedMatrix, aucMaxRank: Optional[float] = None, *, ctx=None, out=None):
    """`replaid.aucell(X, matG, aucMaxRank=ceiling(0.05*nrow(X)))` (R/plaid.R:304-309)."""
    a = float(aucMaxRank) if aucMaxRank is not None else float(math.ceil(0.05 * X.shape[0]))
    return _score(X, matG, dict(scorer=L.AUCELL, auc_max_rank=a), ctx, out)


def replaid_gsva(X: NamedMatrix, matG: NamedMatrix, tau: float = 0.0, rowtf: str = "z", *, ctx=None, out=None):
    """`replaid.gsva(X, matG, tau=0, rowtf="z")` (R/plaid.R:338-363).  `rowtf="ecdf"` ranks every gene
    ACROSS the samples of the call (single shard: it needs all samples); any other value is the reference's error."""
    if isinstance(rowtf, (list, tuple)):
        rowtf = rowtf[0]
    if rowtf not in ("z", "ecdf"):
        raise ValueError("Error: unknown row transform" + str(rowtf))  # R/plaid.R:348
    return _score(X, matG, dict(scorer=L.GSVA, tau=float(tau), gsva_ecdf=1 if rowtf == "ecdf" else 0), ctx, out)


# ---------------------------------------------------------------------------------------
# plaid.test: the reductions run on the GPU, the distribution functions stay on the host (as stats::pt does in R)
# ---------------------------------------------------------------------------------------
def group_moments(gsetX, y, *, ctx=None):
    """Per row of a dense S x N matrix: (sum, sum of squares) over the columns with y == 0 and with y == 1
    (`plaidgpu_group_moments`); the reductions of Rfast::ttests in plaid.test (R/plaid.R:429-431)."""
    ctx = ctx or default_context()
    y32 = np.ascontiguousarray(np.asarray(y), dtype=np.int32)
    if _is_torch(gsetX):
        raise TypeError("pass device matrices through the C ABI directly")
    a = np.asfortranarray(np.asarray(gsetX, dtype=np.float64))
    out = np.empty((4, a.shape[0]), dtype=np.float64)
    ctx.check(ctx.lib.plaidgpu_group_moments(ctx.h, a.ctypes.data, a.shape[0], a.shape[1], y32.ctypes.data, L.HOST,
                                             out.ctypes.data))
    return out


def score_group_moments(X: NamedMatrix, matG: NamedMatrix, y, *, ctx=None, **opts_kw):
    """plaid() (or another scorer through `opts_kw`) fused with the group reductions of plaid.test(tests="lm")
    (`plaidgpu_score_group_moments`, R/plaid.R:423-431): the S x N score matrix stays on the device as raw scores,
    the normalisation is applied in registers while reducing, 4 x S doubles come back.  Returns (4, S) like
    group_moments, or None on no overlap."""
    ctx = ctx or default_context()
    if X.rownames is None or matG.rownames is None:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    rowmap = make_rowmap(X.rownames, matG.rownames)
    if not (rowmap >= 0).any():
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.set_genesets(matG.mat)
    keep: list = []
    M = _matrix_struct(X.mat, keep)
    y32 = np.ascontiguousarray(np.asarray(y), dtype=np.int32)
    if y32.size != M.N:
        raise ValueError("length(y) must equal ncol(X)")
    kw = dict(scorer=L.PLAID, stats_mean=1, normalize=1)
    kw.update(opts_kw)
    o = _opts(ctx.lib, **kw)
    out = np.empty((4, int(matG.mat.shape[1])), dtype=np.float64)
    rc = ctx.lib.plaidgpu_score_group_moments(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), y32.ctypes.data,
                                              out.ctypes.data)
    if rc == L.ERR_NOOVERLAP:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.check(rc)
    return out


def group_stats(gsetX, labels, K=None, *, ctx=None):
    """Per row of a dense S x N matrix: (sum, sum of squares) over the columns of each group k = labels[j] in [0, K)
    (`plaidgpu_group_stats`); a label of -1 leaves the column out.  K defaults to max(labels) + 1.  Returns an
    array of shape (K, 2, S); empty groups give zeros."""
    ctx = ctx or default_context()
    if _is_torch(gsetX):
        raise TypeError("pass device matrices through the C ABI directly")
    a = np.asfortranarray(np.asarray(gsetX, dtype=np.float64))
    lab, K = _labels(labels, a.shape[1], K)
    out = np.empty((K, 2, a.shape[0]), dtype=np.float64)
    ctx.check(ctx.lib.plaidgpu_group_stats(ctx.h, a.ctypes.data, a.shape[0], a.shape[1], lab.ctypes.data, K, L.HOST,
                                           out.ctypes.data))
    return out


def _labels(labels, n, K):
    lab = np.ascontiguousarray(np.asarray(labels), dtype=np.int32)
    if lab.ndim != 1 or lab.size != n:
        raise ValueError("length(labels) must equal ncol(X)")
    if K is None:
        K = int(lab.max()) + 1 if lab.size else 1
    return lab, int(K)


def score_group_stats(X: NamedMatrix, matG: NamedMatrix, labels, K=None, *, ctx=None, **opts_kw):
    """plaid() (or another scorer through `opts_kw`) fused with the per-group reductions of group_stats
    (`plaidgpu_score_group_stats`): the S x N scores stay on the device, K x 2 x S doubles come back.  `ctx` may be a
    list of Contexts on different devices: the columns are then split over them
    (`plaidgpu_score_group_stats_multi`).  Returns an array of shape (K, 2, S), or None on no overlap."""
    ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else None
    ctx = (ctxs[0] if ctxs else ctx) or default_context()
    if X.rownames is None or matG.rownames is None:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    rowmap = make_rowmap(X.rownames, matG.rownames)
    if not (rowmap >= 0).any():
        _message("[plaid] ERROR. No overlapping features.")
        return None
    for cx in (ctxs or [ctx]):
        cx.set_genesets(matG.mat)
    keep: list = []
    M = _matrix_struct(X.mat, keep)
    lab, K = _labels(labels, M.N, K)
    kw = dict(scorer=L.PLAID, stats_mean=1, normalize=1)
    kw.update(opts_kw)
    o = _opts(ctx.lib, **kw)
    out = np.empty((K, 2, int(matG.mat.shape[1])), dtype=np.float64)
    if ctxs and len(ctxs) > 1:
        hs = (C.c_void_p * len(ctxs))(*[cx.h for cx in ctxs])
        rc = ctx.lib.plaidgpu_score_group_stats_multi(hs, len(ctxs), C.byref(M), rowmap.ctypes.data, C.byref(o),
                                                      lab.ctypes.data, K, out.ctypes.data)
    else:
        rc = ctx.lib.plaidgpu_score_group_stats(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), lab.ctypes.data, K,
                                                out.ctypes.data)
    if rc == L.ERR_NOOVERLAP:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.check(rc)
    return out


def _dense_input(gsetX):
    """(S, N, location, pointer, keep) of a dense S x N matrix given as a 2-D array or a DeviceDense"""
    if isinstance(gsetX, DeviceDense):
        S, N = (int(d) for d in gsetX.shape)
        if gsetX.x.numel() != S * N:
            raise ValueError("DeviceDense: the tensor does not hold shape[0] * shape[1] values")
        return S, N, L.DEVICE, gsetX.x.data_ptr(), gsetX
    if _is_torch(gsetX):
        raise TypeError("pass dense device matrices as DeviceDense(t_colmajor, shape)")
    a = np.asarray(gsetX, dtype=np.float64)
    if a.ndim != 2:
        raise ValueError("gsetX must be a matrix (S x N)")
    a = np.asfortranarray(a)
    return a.shape[0], a.shape[1], L.HOST, a.ctypes.data, a


def col_topk(gsetX, k=10, decreasing=True, *, ctx=None):
    """Per column of a dense S x N matrix: the first k entries of R's `order(v, decreasing = decreasing)`, i.e. the
    k largest (or smallest) values with ties by ascending row and NaN last (`plaidgpu_col_topk`).  `gsetX` is a 2-D
    array or a `DeviceDense` (S x N in device memory).  Returns (idx, val) of shape (k, N): 0-based row indices
    (int32) and the values at those rows, bit for bit."""
    ctx = ctx or default_context()
    S, N, loc, ptr, keep = _dense_input(gsetX)
    idx = np.empty((max(int(k), 0), N), dtype=np.int32, order="F")  # a bad k is the library's error
    val = np.empty((max(int(k), 0), N), dtype=np.float64, order="F")
    ctx.check(ctx.lib.plaidgpu_col_topk(ctx.h, ptr, S, N, int(k), 1 if decreasing else 0, loc, idx.ctypes.data,
                                        val.ctypes.data))
    del keep
    return idx, val


def score_topk(X: NamedMatrix, matG: NamedMatrix, k=10, decreasing=True, *, ctx=None, **opts_kw):
    """plaid() (or another scorer through `opts_kw`) fused with col_topk (`plaidgpu_score_topk`): each cell's k
    best gene sets, while the S x N scores stay on the device.  Equal, bit for bit, to scoring followed by col_topk.
    `ctx` may be a list of Contexts on different devices: the columns are then split over them
    (`plaidgpu_score_topk_multi`).  Returns (idx, val) of shape (k, N), or None on no overlap."""
    ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else None
    ctx = (ctxs[0] if ctxs else ctx) or default_context()
    if X.rownames is None or matG.rownames is None:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    rowmap = make_rowmap(X.rownames, matG.rownames)
    if not (rowmap >= 0).any():
        _message("[plaid] ERROR. No overlapping features.")
        return None
    for cx in (ctxs or [ctx]):
        cx.set_genesets(matG.mat)
    keep: list = []
    M = _matrix_struct(X.mat, keep)
    kw = dict(scorer=L.PLAID, stats_mean=1, normalize=1)
    kw.update(opts_kw)
    o = _opts(ctx.lib, **kw)
    idx = np.empty((max(int(k), 0), M.N), dtype=np.int32, order="F")
    val = np.empty((max(int(k), 0), M.N), dtype=np.float64, order="F")
    dec = 1 if decreasing else 0
    if ctxs and len(ctxs) > 1:
        hs = (C.c_void_p * len(ctxs))(*[cx.h for cx in ctxs])
        rc = ctx.lib.plaidgpu_score_topk_multi(hs, len(ctxs), C.byref(M), rowmap.ctypes.data, C.byref(o), int(k), dec,
                                               idx.ctypes.data, val.ctypes.data)
    else:
        rc = ctx.lib.plaidgpu_score_topk(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), int(k), dec,
                                         idx.ctypes.data, val.ctypes.data)
    if rc == L.ERR_NOOVERLAP:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.check(rc)
    return idx, val


def row_topk(gsetX, k=10, decreasing=True, *, ctx=None):
    """Per row of a dense S x N matrix: the first k entries of R's `order(x[s, ], decreasing = decreasing)`, i.e. the
    k largest (or smallest) values with ties by ascending column and NaN last (`plaidgpu_row_topk`).  `gsetX` is a 2-D
    array or a `DeviceDense` (S x N in device memory).  Returns (idx, val) of shape (k, S): 0-based column indices
    (int64) and the values at those columns, bit for bit."""
    ctx = ctx or default_context()
    S, N, loc, ptr, keep = _dense_input(gsetX)
    idx = np.empty((max(int(k), 0), S), dtype=np.int64, order="F")  # a bad k is the library's error
    val = np.empty((max(int(k), 0), S), dtype=np.float64, order="F")
    ctx.check(ctx.lib.plaidgpu_row_topk(ctx.h, ptr, S, N, int(k), 1 if decreasing else 0, loc, idx.ctypes.data,
                                        val.ctypes.data))
    del keep
    return idx, val


def score_row_topk(X: NamedMatrix, matG: NamedMatrix, k=10, decreasing=True, *, ctx=None, **opts_kw):
    """plaid() (or another scorer through `opts_kw`) fused with row_topk (`plaidgpu_score_row_topk`): each gene set's
    k best cells, while the S x N scores stay on the device.  Equal, bit for bit, to scoring followed by row_topk.
    `ctx` may be a list of Contexts on different devices: the columns are then split over them and the lists merged
    (`plaidgpu_score_row_topk_multi`).  Returns (idx, val) of shape (k, S), or None on no overlap."""
    ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else None
    ctx = (ctxs[0] if ctxs else ctx) or default_context()
    if X.rownames is None or matG.rownames is None:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    rowmap = make_rowmap(X.rownames, matG.rownames)
    if not (rowmap >= 0).any():
        _message("[plaid] ERROR. No overlapping features.")
        return None
    for cx in (ctxs or [ctx]):
        cx.set_genesets(matG.mat)
    keep: list = []
    M = _matrix_struct(X.mat, keep)
    kw = dict(scorer=L.PLAID, stats_mean=1, normalize=1)
    kw.update(opts_kw)
    o = _opts(ctx.lib, **kw)
    S = int(matG.mat.shape[1])
    idx = np.empty((max(int(k), 0), S), dtype=np.int64, order="F")
    val = np.empty((max(int(k), 0), S), dtype=np.float64, order="F")
    dec = 1 if decreasing else 0
    if ctxs and len(ctxs) > 1:
        hs = (C.c_void_p * len(ctxs))(*[cx.h for cx in ctxs])
        rc = ctx.lib.plaidgpu_score_row_topk_multi(hs, len(ctxs), C.byref(M), rowmap.ctypes.data, C.byref(o), int(k),
                                                   dec, idx.ctypes.data, val.ctypes.data)
    else:
        rc = ctx.lib.plaidgpu_score_row_topk(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), int(k), dec,
                                             idx.ctypes.data, val.ctypes.data)
    if rc == L.ERR_NOOVERLAP:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.check(rc)
    return idx, val


def _design_basis(B, n):
    b = np.asarray(B, dtype=np.float64)
    if b.ndim == 1:
        b = b[:, None]
    if b.ndim != 2 or b.shape[0] != n:
        raise ValueError("nrow(B) must equal ncol(X)")
    return np.asfortranarray(b)  # a bad Q or a non-finite entry is the library's error


def design_stats(gsetX, B, *, ctx=None):
    """Per row s of a dense S x N matrix x: sum_j x[s, j] * B[j, q] for every column q of the N x Q matrix B
    (1 <= Q <= 64, finite), then sum_j x[s, j] and sum_j x[s, j]^2 (`plaidgpu_design_stats`): the reductions behind
    plaid_lm, one pass over x.  `gsetX` is a 2-D array or a `DeviceDense`.  Returns an array of shape (Q + 2, S)."""
    ctx = ctx or default_context()
    S, N, loc, ptr, keep = _dense_input(gsetX)
    b = _design_basis(B, N)
    out = np.empty((b.shape[1] + 2, S), dtype=np.float64)
    ctx.check(ctx.lib.plaidgpu_design_stats(ctx.h, ptr, S, N, b.ctypes.data, b.shape[1], loc, out.ctypes.data))
    del keep
    return out


def score_design_stats(X: NamedMatrix, matG: NamedMatrix, B, *, ctx=None, **opts_kw):
    """plaid() (or another scorer through `opts_kw`) fused with design_stats (`plaidgpu_score_design_stats`): the S x N
    scores stay on the device, (Q + 2) x S doubles come back.  B: N x Q, one row per column of X.  `ctx` may be a list
    of Contexts on different devices: the columns are then split over them (`plaidgpu_score_design_stats_multi`).
    Returns an array of shape (Q + 2, S), or None on no overlap."""
    ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else None
    ctx = (ctxs[0] if ctxs else ctx) or default_context()
    if X.rownames is None or matG.rownames is None:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    rowmap = make_rowmap(X.rownames, matG.rownames)
    if not (rowmap >= 0).any():
        _message("[plaid] ERROR. No overlapping features.")
        return None
    for cx in (ctxs or [ctx]):
        cx.set_genesets(matG.mat)
    keep: list = []
    M = _matrix_struct(X.mat, keep)
    b = _design_basis(B, M.N)
    kw = dict(scorer=L.PLAID, stats_mean=1, normalize=1)
    kw.update(opts_kw)
    o = _opts(ctx.lib, **kw)
    out = np.empty((b.shape[1] + 2, int(matG.mat.shape[1])), dtype=np.float64)
    if ctxs and len(ctxs) > 1:
        hs = (C.c_void_p * len(ctxs))(*[cx.h for cx in ctxs])
        rc = ctx.lib.plaidgpu_score_design_stats_multi(hs, len(ctxs), C.byref(M), rowmap.ctypes.data, C.byref(o),
                                                       b.ctypes.data, b.shape[1], out.ctypes.data)
    else:
        rc = ctx.lib.plaidgpu_score_design_stats(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), b.ctypes.data,
                                                 b.shape[1], out.ctypes.data)
    if rc == L.ERR_NOOVERLAP:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.check(rc)
    return out


LM_COLUMNS = ["logFC", "SE", "AveExpr", "t", "P.Value", "adj.P.Val"]


def design_qr(design):
    """Thin QR D = U R of an N x Q design (U: N x Q with orthonormal columns, R: Q x Q upper triangular).  Raises
    ValueError for a non-finite entry, Q outside [1, 64], or a design that is not of full column rank (a column whose
    part orthogonal to the columns before it is below 1e-7 of its norm, the tolerance of R's qr())."""
    D = np.asarray(design, dtype=np.float64)
    if D.ndim == 1:
        D = D[:, None]
    if D.ndim != 2 or not 1 <= D.shape[1] <= 64:
        raise ValueError("the design must be a matrix with 1 to 64 columns")
    if not np.all(np.isfinite(D)):
        raise ValueError("the design must be finite (no NA)")
    if D.shape[0] < D.shape[1]:
        raise ValueError("the design is not of full column rank")
    U, R = np.linalg.qr(D)
    if np.any(np.abs(np.diag(R)) <= 1e-7 * np.linalg.norm(D, axis=0)):
        raise ValueError("the design is not of full column rank")
    return U, R


def _bh(p):
    """p.adjust(p, "BH"); NaN stays NaN and does not count"""
    q = np.full(p.shape, np.nan)
    ok = ~np.isnan(p)
    pv = p[ok]
    n = pv.size
    if n:
        o = np.argsort(-pv, kind="stable")
        q[ok] = np.minimum(1.0, np.minimum.accumulate((n / np.arange(n, 0, -1)) * pv[o]))[np.argsort(o, kind="stable")]
    return q


def lm_from_moments(mom, R, N, contrasts=None):
    """Ordinary least squares of every gene set's N scores on a design D = U R, from the moments design_stats(x, U)
    returns (z = U^T x_s, a = sum x_s, t = sum x_s^2, per set): beta = R^-1 z, RSS = max(t - |z|^2, 0), df = N - Q,
    sigma^2 = RSS / df; per contrast vector c (a column of `contrasts`, Q x L; None = the coefficients themselves):
    logFC = c^T beta, SE = sigma |R^-T c|, t = logFC / SE, P.Value = 2 pt(-|t|, df), adj.P.Val = BH over the sets,
    AveExpr = a / N.  SE, t and P.Value are NaN when df <= 0 or sigma = 0; a set with a NaN score gives NaN throughout.
    Returns one S x 6 table per contrast, columns LM_COLUMNS."""
    from scipy import linalg, stats
    R = np.asarray(R, dtype=np.float64)
    Q = R.shape[0]
    mom = np.asarray(mom, dtype=np.float64)
    if mom.ndim != 2 or mom.shape[0] != Q + 2:
        raise ValueError("the moments must have Q + 2 rows")
    Cm = np.eye(Q) if contrasts is None else np.asarray(contrasts, dtype=np.float64)
    if Cm.ndim == 1:
        Cm = Cm[:, None]
    if Cm.ndim != 2 or Cm.shape[0] != Q:
        raise ValueError("the contrasts must have one row per column of the design")
    z, a, t2 = mom[:Q], mom[Q], mom[Q + 1]
    df = N - Q
    with np.errstate(invalid="ignore", divide="ignore"):
        beta = linalg.solve_triangular(R, z, check_finite=False)
        rss = np.maximum(t2 - (z * z).sum(axis=0), 0.0)
        sigma = np.sqrt(rss / df) if df > 0 else np.full(a.shape, np.nan)
        sefac = np.sqrt((linalg.solve_triangular(R, Cm, trans="T") ** 2).sum(axis=0))
        tabs = []
        for l in range(Cm.shape[1]):
            logfc = Cm[:, l] @ beta
            se = sigma * sefac[l]
            se[(sigma == 0)] = np.nan
            tt = logfc / se
            p = 2.0 * stats.t.sf(np.abs(tt), df) if df > 0 else np.full(a.shape, np.nan)
            tabs.append(np.column_stack([logfc, se, a / N, tt, p, _bh(p)]))
    return tabs


def _named_columns(m, prefix):
    if isinstance(m, NamedMatrix):
        a = np.asarray(m.mat, dtype=np.float64)
        names = m.colnames
    else:
        a, names = np.asarray(m, dtype=np.float64), None
    if a.ndim == 1:
        a = a[:, None]
    if names is None:
        names = [f"{prefix}{k + 1}" for k in range(a.shape[1] if a.ndim == 2 else 0)]
    return a, list(names)


def plaid_lm(X: NamedMatrix, G: NamedMatrix, design, contrasts=None, gsetX: Optional[NamedMatrix] = None,
             sort_by: str = "none", *, ctx=None, **opts_kw):
    """Ordinary least squares of every gene set's plaid scores on `design` (N x Q, one row per column of X, finite,
    full column rank, 1 <= Q <= 64): R's lm(gsetX[s, ] ~ design - 1) for every set s, or limma's lmFit +
    contrasts.fit without eBayes.  `design` / `contrasts` (Q x L) are arrays or NamedMatrix (their colnames name the
    results; otherwise coef1.. / contrast1..).  The host takes a thin QR D = U R; the GPU returns U^T x_s, sum x_s and
    sum x_s^2 per set, fused onto the scoring call (score_design_stats; `opts_kw` selects another scorer, a list of
    Contexts splits the columns) or from gsetX (design_stats); lm_from_moments does the rest.  A NaN score makes that
    set's statistics NaN (lm would drop the sample instead).  Returns {name: (table, LM_COLUMNS, set names)}, tables
    sorted by `sort_by` when it names a column, or None on no overlap."""
    ctx0 = (ctx[0] if isinstance(ctx, (list, tuple)) else ctx) or default_context()
    D, coef = _named_columns(design, "coef")
    if D.ndim != 2 or D.shape[0] != X.shape[1]:
        raise ValueError("nrow(design) must equal ncol(X)")
    U, R = design_qr(D)
    Cm, names = (None, coef) if contrasts is None else _named_columns(contrasts, "contrast")
    if Cm is not None and (Cm.ndim != 2 or Cm.shape[0] != D.shape[1]):
        raise ValueError("nrow(contrasts) must equal ncol(design)")
    if gsetX is None:
        mom = score_design_stats(X, G, U, ctx=ctx, **opts_kw)
        if mom is None:
            return None
    else:
        mom = design_stats(gsetX.mat if isinstance(gsetX, NamedMatrix) else gsetX, U, ctx=ctx0)
    tabs = lm_from_moments(mom, R, D.shape[0], Cm)
    rows = list(G.colnames) if G.colnames is not None else [str(k) for k in range(mom.shape[1])]
    res = {}
    for name, tab in zip(names, tabs):
        r = rows
        if sort_by in LM_COLUMNS:
            o = np.argsort(tab[:, LM_COLUMNS.index(sort_by)], kind="stable")
            tab, r = tab[o], [rows[k] for k in o]
        res[name] = (tab, list(LM_COLUMNS), r)
    return res


def _align(X: NamedMatrix, G: NamedMatrix):
    """intersect(rownames(G), rownames(X)) and X[gg, ], G[gg, ] (R/plaid.R:402-404)"""
    xset = set(X.rownames)
    gg = [g for g in dict.fromkeys(G.rownames) if g in xset]
    xpos, gpos = {}, {}
    for k, n in enumerate(X.rownames):
        xpos.setdefault(n, k)
    for k, n in enumerate(G.rownames):
        gpos.setdefault(n, k)
    xi = np.array([xpos[g] for g in gg])
    gi = np.array([gpos[g] for g in gg])
    Xs = sp.csc_matrix(X.mat).tocsr()[xi].tocsc() if sp.issparse(X.mat) else np.asarray(X.mat, dtype=np.float64)[xi]
    Gs = sp.csc_matrix(G.mat).tocsr()[gi].tocsc()
    Gb = Gs.copy()
    Gb.data = (Gb.data != 0).astype(np.float64)
    Gb.eliminate_zeros()
    return gg, Xs, Gs, Gb


def _set_tests(tests, s1, q1, sumG, ngenes, fc, P, Fs):
    """the "one" and "two" tests of plaid.test from crossprod(G != 0, [fc, fc^2]) = [s1, q1] (R/plaid.R:476-520)"""
    from scipy import stats
    with np.errstate(invalid="ignore", divide="ignore"):
        if "one" in tests:  # R/plaid.R:476-486
            meanx = s1 / (1e-8 + sumG)
            sdx = np.sqrt((q1 - meanx ** 2 * sumG) / (sumG - 1))
            t = meanx / (1e-8 + sdx) * np.sqrt(sumG)
            P["one"], Fs["one"] = 2.0 * stats.t.sf(np.abs(t), np.maximum(sumG - 1, 1)), meanx
        if "two" in tests:  # R/plaid.R:488-520
            sum1, sum0 = sumG, ngenes - sumG
            ssq0, m0 = -q1 + (fc ** 2).sum(), -s1 + fc.sum()
            mean1, mean0 = s1 / (1e-8 + sum1), m0 / (1e-8 + sum0)
            var0 = (ssq0 - mean0 ** 2 * sum0) / (sum0 - 1)
            var1 = (q1 - mean1 ** 2 * sum1) / (sum1 - 1)
            varsum = var0 / sum0 + var1 / sum1
            dof = varsum ** 2 / (var0 / sum0 * (sum0 - 1) + var1 / sum1 * (sum1 - 1))
            f = mean1 - mean0
            P["two"], Fs["two"] = 2.0 * stats.t.sf(np.abs(f / np.sqrt(varsum)), np.maximum(dof, 1)), f


def _lm_test(s0, q0, n0, s1, q1, n1, P, Fs):
    """Rfast::ttests(t(gsetX), ina = y + 1) (R/plaid.R:429-431) from the group sums / sums of squares: Welch's test
    of group 1 against group 0"""
    from scipy import stats
    with np.errstate(invalid="ignore", divide="ignore"):
        m1, m2 = s0 / n0, s1 / n1  # ina 1 = (y == 0), ina 2 = (y == 1)
        v1 = (q0 - n0 * m1 ** 2) / (n0 - 1)
        v2 = (q1 - n1 * m2 ** 2) / (n1 - 1)
        fac = v1 / n0 + v2 / n1
        stat = (m1 - m2) / np.sqrt(fac)
        dof = fac ** 2 / ((v1 / n0) ** 2 / (n0 - 1) + (v2 / n1) ** 2 / (n1 - 1))
        P["lm"], Fs["lm"] = 2.0 * stats.t.sf(np.abs(stat), dof), m2 - m1


def _test_table(P, Fs, G: NamedMatrix, metap_method, sort_by):
    """p-value clamp, meta p-value, FDR and the sorted result table of plaid.test (R/plaid.R:440-474)"""
    from scipy import stats
    for k in P:
        p1 = np.where(np.isnan(P[k]), 1.0, P[k])
        P[k] = np.minimum(np.maximum(p1, 1e-99), 1 - 1e-99)
    keys = [k for k in ("one", "two", "lm") if k in P]
    gsetFC = np.column_stack([Fs[k] for k in keys]).mean(axis=1)
    if len(keys) > 1:
        if metap_method in ("fisher", "sumlog"):
            pmeta = stats.chi2.sf(-2.0 * sum(np.log(P[k]) for k in keys), 2 * len(keys))
        elif metap_method in ("stouffer", "sumz"):
            pmeta = stats.norm.sf(sum(stats.norm.isf(P[k]) for k in keys) / math.sqrt(len(keys)))
        else:
            raise ValueError("Invalid method: " + metap_method)
    else:
        pmeta = P[keys[0]]
    n = pmeta.size  # p.adjust(method = "fdr")
    o = np.argsort(-pmeta, kind="stable")
    q = np.minimum(np.minimum.accumulate(pmeta[o] * n / np.arange(n, 0, -1)), 1.0)[np.argsort(o, kind="stable")]
    cols = ["gsetFC"] + ["p." + k for k in keys] + ["p.meta", "q.meta"]
    tab = np.column_stack([gsetFC] + [P[k] for k in keys] + [pmeta, q])
    rows = list(G.colnames) if G.colnames is not None else [str(k) for k in range(tab.shape[0])]
    if sort_by in cols:
        oo = np.argsort(tab[:, cols.index(sort_by)], kind="stable")
        tab, rows = tab[oo], [rows[k] for k in oo]
    return tab, cols, rows


def plaid_test(X: NamedMatrix, y, G: NamedMatrix, gsetX: Optional[NamedMatrix] = None, tests=("one", "two", "lm"),
               metap_method: str = "fisher", sort_by: str = "p.meta", *, ctx=None):
    """`plaid.test(X, y, G, gsetX, tests=c("one","two","lm"), metap.method="fisher", sort.by="p.meta")`
    (R/plaid.R:392-474).  GPU: the score matrix (plaid), the crossprods of the one/two-sample tests
    (chunked_crossprod on G != 0) and the per-set group moments of the "lm" test; host: pt / pchisq / p.adjust.
    Returns (table, column names, row names) like the oracle."""
    ctx = ctx or default_context()
    y = np.asarray(y)
    if not np.all(np.isin(np.unique(y), [0, 1])):
        raise ValueError("elements of y must be 0 or 1")  # R/plaid.R:394
    gg, Xs, Gs, Gb = _align(X, G)
    n1, n0 = int((y == 1).sum()), int((y == 0).sum())
    if sp.issparse(Xs):
        fc = np.asarray(Xs[:, y == 1].sum(axis=1)).ravel() / n1 - np.asarray(Xs[:, y == 0].sum(axis=1)).ravel() / n0
    else:
        fc = Xs[:, y == 1].mean(axis=1) - Xs[:, y == 0].mean(axis=1)
    sumG = np.asarray(Gb.sum(axis=0)).ravel()
    P, Fs = {}, {}
    if "one" in tests or "two" in tests:
        cp = chunked_crossprod(Gb, np.column_stack([fc, fc ** 2]), ctx=ctx)  # crossprod(G != 0, [F, F^2]) on the GPU
        _set_tests(tests, cp[:, 0], cp[:, 1], sumG, Gb.shape[0], fc, P, Fs)
    if "lm" in tests:  # R/plaid.R:423-433
        if gsetX is None:  # scores never leave the device: reductions fused onto the scoring call
            _message("[plaid.test] computing plaid scores...")
            gm = score_group_moments(NamedMatrix(Xs, gg, X.colnames), NamedMatrix(Gs, gg, G.colnames), y, ctx=ctx)
        else:
            gm = group_moments(gsetX.mat, y, ctx=ctx)
        _lm_test(gm[0], gm[1], n0, gm[2], gm[3], n1, P, Fs)
    return _test_table(P, Fs, G, metap_method, sort_by)


def _missing(v) -> bool:
    return v is None or v != v  # None or NaN


def plaid_test_groups(X: NamedMatrix, groups, G: NamedMatrix, gsetX: Optional[NamedMatrix] = None,
                      tests=("one", "two", "lm"), metap_method: str = "fisher", sort_by: str = "p.meta", *, ctx=None):
    """plaid_test of every group against all other labelled cells, in one scoring pass.  `groups` holds one label per
    cell of X; None / NaN leaves the cell out.  Returns {label: (table, column names, row names)} over the sorted
    unique labels, each entry what `plaid_test(X[:, keep], groups[keep] == label, G, gsetX[:, keep])` returns with
    keep = the labelled cells.  GPU: the scores and their per-group moments (score_group_stats, or group_stats on
    gsetX) and one crossprod(G != 0, [F_1..F_K, F_1^2..F_K^2]); host: the per-group gene means (one sparse product)
    and the distribution functions.  `ctx` may be a list of Contexts (the scores are then split over them)."""
    ctx0 = (ctx[0] if isinstance(ctx, (list, tuple)) else ctx) or default_context()
    groups = list(groups)
    if len(groups) != X.shape[1]:
        raise ValueError("length(groups) must equal ncol(X)")
    keep = np.array([not _missing(v) for v in groups], dtype=bool)
    levels = sorted(set(v for v, k in zip(groups, keep) if k))
    if not levels:
        raise ValueError("no cell has a group label")
    index = {v: k for k, v in enumerate(levels)}
    labels = np.array([index[v] if k else -1 for v, k in zip(groups, keep)], dtype=np.int32)
    K = len(levels)
    lab = labels[keep]
    n = int(lab.size)
    nk = np.bincount(lab, minlength=K).astype(np.float64)
    gg, Xs, Gs, Gb = _align(X, G)
    Xs = Xs[:, np.flatnonzero(keep)]
    colnames = [X.colnames[j] for j in np.flatnonzero(keep)] if X.colnames is not None else None
    P = [dict() for _ in range(K)]
    Fs = [dict() for _ in range(K)]
    with np.errstate(invalid="ignore", divide="ignore"):
        if "one" in tests or "two" in tests:
            onehot = sp.csc_matrix((np.ones(n), (np.arange(n), lab)), shape=(n, K))
            gsum = np.asarray((Xs @ onehot).todense() if sp.issparse(Xs) else Xs @ onehot.toarray())  # genes x K
            total = np.asarray(Xs.sum(axis=1)).ravel()
            F = gsum / nk - (total[:, None] - gsum) / (n - nk)  # mean(group) - mean(other labelled cells)
            alone = nk == n  # no other cell: F is NaN, and so is every statistic built on it
            Fz = np.where(alone, 0.0, F)
            cp = chunked_crossprod(Gb, np.column_stack([Fz, Fz ** 2]), ctx=ctx0)  # crossprod(G != 0, [F_k, F_k^2])
            cp[:, np.concatenate([alone, alone])] = np.nan
            sumG = np.asarray(Gb.sum(axis=0)).ravel()
            for k in range(K):
                _set_tests(tests, cp[:, k], cp[:, K + k], sumG, Gb.shape[0], F[:, k], P[k], Fs[k])
        if "lm" in tests:
            if gsetX is None:
                _message("[plaid.test] computing plaid scores...")
                gm = score_group_stats(NamedMatrix(Xs, gg, colnames), NamedMatrix(Gs, gg, G.colnames), lab, K, ctx=ctx)
            else:
                gm = group_stats(gsetX.mat, labels, K, ctx=ctx0)
            tot = gm.sum(axis=0)  # all labelled cells: (2, S)
            for k in range(K):
                _lm_test(tot[0] - gm[k, 0], tot[1] - gm[k, 1], n - nk[k], gm[k, 0], gm[k, 1], nk[k], P[k], Fs[k])
    return {levels[k]: _test_table(P[k], Fs[k], G, metap_method, sort_by) for k in range(K)}


# ---------------------------------------------------------------------------------------
# gene-set ingestion (host-side C++ behind the same ABI; needs no GPU)
# ---------------------------------------------------------------------------------------
def gmt2mat_file(path: str) -> NamedMatrix:
    """`gmt2mat(read.gmt(path))` (R/gmt-utils.R:99-125, 19-66) in one call: genes x sets csc_matrix of ones
    with gmt2mat's row / column order."""
    lib = L.load()
    h = C.c_void_p()
    rc = lib.plaidgpu_gmt_read(path.encode(), C.byref(h))
    if rc != L.OK:
        raise L.PlaidGpuError(rc, f"cannot read GMT file {path!r}")
    try:
        S, P, nnz = lib.plaidgpu_gmt_num_sets(h), lib.plaidgpu_gmt_num_genes(h), lib.plaidgpu_gmt_nnz(h)
        gp = np.empty(S + 1, dtype=np.int32)
        gi = np.empty(max(nnz, 1), dtype=np.int32)
        rc = lib.plaidgpu_gmt_csc(h, gp.ctypes.data, gi.ctypes.data)
        if rc != L.OK:
            raise L.PlaidGpuError(rc, "plaidgpu_gmt_csc failed")
        sets = [lib.plaidgpu_gmt_set_name(h, k).decode() for k in range(S)]
        genes = [lib.plaidgpu_gmt_gene_name(h, k).decode() for k in range(P)]
        G = sp.csc_matrix((np.ones(nnz), gi[:nnz], gp), shape=(P, S))
        return NamedMatrix(G, genes, sets)
    finally:
        lib.plaidgpu_gmt_free(h)


# ---------------------------------------------------------------------------------------
# expression-matrix files and tiled result egress (scope row f4; readers need no GPU)
# ---------------------------------------------------------------------------------------
def _spmat_to_named(lib, h) -> NamedMatrix:
    try:
        M = L.Matrix()
        rc = lib.plaidgpu_spmat_view(h, C.byref(M))
        if rc != L.OK:
            raise L.PlaidGpuError(rc, "plaidgpu_spmat_view failed")
        nnz = lib.plaidgpu_spmat_nnz(h)
        p = np.ctypeslib.as_array(C.cast(M.p, C.POINTER(C.c_int32)), shape=(M.N + 1,)).copy()
        if nnz:
            i = np.ctypeslib.as_array(C.cast(M.i, C.POINTER(C.c_int32)), shape=(nnz,)).copy()
            x = np.ctypeslib.as_array(C.cast(M.x, C.POINTER(C.c_double)), shape=(nnz,)).copy()
        else:
            i, x = np.zeros(0, dtype=np.int32), np.zeros(0)
        rn = [lib.plaidgpu_spmat_rowname(h, k).decode() for k in range(lib.plaidgpu_spmat_num_rownames(h))] or None
        cn = [lib.plaidgpu_spmat_colname(h, k).decode() for k in range(lib.plaidgpu_spmat_num_colnames(h))] or None
        return NamedMatrix(sp.csc_matrix((x, i, p), shape=(M.P, M.N)), rn, cn)
    finally:
        lib.plaidgpu_spmat_free(h)


def _read_spmat(fn_name: str, *args) -> NamedMatrix:
    lib = L.load()
    h = C.c_void_p()
    rc = getattr(lib, fn_name)(*args, C.byref(h))
    if rc != L.OK:
        raise L.PlaidGpuError(rc, lib.plaidgpu_io_error().decode(errors="replace"))
    return _spmat_to_named(lib, h)


def read_rda(path: str, name: Optional[str] = None) -> NamedMatrix:
    """`load(path)` / `readRDS(path)` for a file holding a `dgCMatrix` (the reference's fixture format,
    inst/extdata/pbmc3k-50cells.rda, dev/extdata.R:15): the sparse matrix with its dimnames."""
    return _read_spmat("plaidgpu_spmat_read_rda", path.encode(), name.encode() if name else None)


def read_mtx(path: str) -> NamedMatrix:
    """`as(Matrix::readMM(path), "CsparseMatrix")` for Matrix Market coordinate files (plain or .gz)."""
    return _read_spmat("plaidgpu_spmat_read_mtx", path.encode())


def read_10x(directory: str) -> NamedMatrix:
    """`Seurat::Read10X(directory)`-style ingestion: matrix.mtx[.gz] + features.tsv / genes.tsv (gene symbols as
    rownames) + barcodes.tsv (colnames).  Names are kept as they are (no make.unique): a duplicated symbol's
    first row is the one that aligns with matG, like `intersect` + `match` in R/plaid.R:65-72."""
    return _read_spmat("plaidgpu_spmat_read_10x", directory.encode())


def score_to_file(X: NamedMatrix, matG: NamedMatrix, path: str, *, fmt: str = "npy", ctx=None, **opts_kw):
    """Score and stream the S x N result to `path` in column tiles (results larger than host memory).
    opts_kw are the plaidgpu_opts fields (default: plaid(), stats = "mean", normalize = TRUE).  Returns (S, N)."""
    ctx = ctx or default_context()
    if X.rownames is None or matG.rownames is None:
        _message("[plaid] ERROR. No overlapping features.")
        return None
    rowmap = make_rowmap(X.rownames, matG.rownames)
    if not (rowmap >= 0).any():
        _message("[plaid] ERROR. No overlapping features.")
        return None
    ctx.set_genesets(matG.mat)
    keep: list = []
    M = _matrix_struct(X.mat, keep)
    o = _opts(ctx.lib, **opts_kw)
    ctx.check(ctx.lib.plaidgpu_score_to_file(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), path.encode(),
                                             L.FILE_NPY if fmt == "npy" else L.FILE_RAW))
    return int(matG.mat.shape[1]), int(M.N)
