"""Per-column top k with set indices (-m gpu): plaidgpu_col_topk against numpy's lexsort on every kind of column
(ties, signed zeros, infinities, NaN, sorted columns), the fused scoring call (plaidgpu_score_topk) against scoring
followed by the selection for seven scorers, the column-tiled route beyond device memory, several contexts and
ThreadComm ranks, a C4-shaped set count, and rejected arguments.  Every comparison is exact: indices equal, values
equal bit for bit (NaN by isnan).  Every test runs twice (fixture `precision`, as in test_gpu_parity.py)."""
import ctypes as C
import threading

import numpy as np
import pytest
import torch

import plaid_b200 as pb
from plaid_b200 import _lib as L, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["tc", "fp64"])
def precision(request):
    from plaid_b200 import api
    old = api.EXACT_FP64
    api.EXACT_FP64 = request.param == "fp64"
    yield request.param
    api.EXACT_FP64 = old


def ref_topk(x, k, decreasing):
    """the first k entries of R's order(v, decreasing = decreasing) for every column v (ties by row, NaN last)"""
    S, N = x.shape
    rows = np.arange(S)
    idx = np.empty((k, N), dtype=np.int32)
    val = np.empty((k, N))
    for j in range(N):
        v = x[:, j]
        o = np.lexsort((rows, -v if decreasing else v, np.isnan(v)))[:k]
        idx[:, j] = o
        val[:, j] = v[o]
    return idx, val


def assert_same(got, want, what=""):
    gi, gv = got
    wi, wv = want
    assert gi.shape == wi.shape and gv.shape == wv.shape, what
    assert np.array_equal(gi, wi), what
    nan = np.isnan(wv)
    assert np.array_equal(np.isnan(gv), nan), what
    assert np.array_equal(gv[~nan].view(np.int64), wv[~nan].view(np.int64)), what


def columns(rng, S, N, kind):
    if kind == "normal":
        return rng.normal(size=(S, N))
    if kind == "ties":
        return rng.integers(-3, 4, size=(S, N)).astype(np.float64)
    if kind == "zeros_inf":  # mixed signed zeros and infinities among a few numbers
        return rng.choice(np.array([0.0, -0.0, np.inf, -np.inf, 1.5, -1.5]), size=(S, N))
    if kind == "some_nan":
        x = rng.normal(size=(S, N))
        x[rng.random((S, N)) < 0.3] = np.nan
        return x
    if kind == "all_nan":
        return np.full((S, N), np.nan)
    if kind == "constant":
        return np.full((S, N), 2.25)
    if kind == "ascending":
        return np.repeat(np.arange(S, dtype=np.float64)[:, None], N, axis=1) + np.arange(N)
    if kind == "descending":
        return np.repeat(-np.arange(S, dtype=np.float64)[:, None], N, axis=1) - np.arange(N)
    raise ValueError(kind)


KINDS = ["normal", "ties", "zeros_inf", "some_nan", "all_nan", "constant", "ascending", "descending"]


@pytest.mark.parametrize("S,N", [(1, 1), (7, 13), (33, 70), (257, 41), (30000, 9)])
def test_col_topk_matches_numpy(S, N, gpu_ctx):
    rng = np.random.default_rng(S * 7 + N)
    ks = sorted({k for k in (1, 31, 32, 33, 255, 256) if k <= S} | ({S} if S <= 256 else set()))
    for kind in KINDS:
        x = columns(rng, S, N, kind)
        xd = torch.from_numpy(np.asfortranarray(x).T.copy()).cuda()  # N x S row-major = S x N column-major
        for k in ks:
            for dec in (True, False):
                want = ref_topk(x, k, dec)
                assert_same(pb.col_topk(x, k, dec, ctx=gpu_ctx), want, (kind, k, dec, "host"))
                assert_same(pb.col_topk(pb.DeviceDense(xd, (S, N)), k, dec, ctx=gpu_ctx), want, (kind, k, dec, "device"))
    assert gpu_ctx.kernel_ms(2) >= 0.0


def test_col_topk_no_columns(gpu_ctx):
    idx, val = pb.col_topk(np.empty((5, 0)), 3, ctx=gpu_ctx)
    assert idx.shape == (3, 0) and val.shape == (3, 0)


@pytest.fixture(scope="module")
def small_case():
    P, N, S = 900, 301, 131
    X = synth.sparse_x_numpy(P, N, seed=201, density=0.3)
    G = synth.genesets_numpy(P, S, seed=202, size_cap=(5, 120))
    names = synth.gene_names(P)
    return pb.NamedMatrix(X, names), pb.NamedMatrix(G, names, synth.set_names(S)), X, G, names


SCORERS = [("plaid", dict(), lambda Xn, Gn, c: pb.plaid(Xn, Gn, ctx=c)),
           ("plaid raw", dict(normalize=0), lambda Xn, Gn, c: pb.plaid(Xn, Gn, normalize=False, ctx=c)),
           ("ucell", dict(scorer=L.UCELL, rmax=200.0), lambda Xn, Gn, c: pb.replaid_ucell(Xn, Gn, rmax=200, ctx=c)),
           ("ssgsea", dict(scorer=L.SSGSEA, alpha=0.0), lambda Xn, Gn, c: pb.replaid_ssgsea(Xn, Gn, ctx=c)),
           ("sing", dict(scorer=L.SING, nrow_x=900), lambda Xn, Gn, c: pb.replaid_sing(Xn, Gn, ctx=c)),
           ("scse", dict(scorer=L.SCSE, remove_log2=-1, score_mean=0), lambda Xn, Gn, c: pb.replaid_scse(Xn, Gn, ctx=c)),
           ("gsva", dict(scorer=L.GSVA, tau=0.0, gsva_ecdf=0), lambda Xn, Gn, c: pb.replaid_gsva(Xn, Gn, ctx=c))]


def test_fused_equals_score_then_select(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    S = Gn.shape[1]
    for name, kw, f in SCORERS:
        full = f(Xn, Gn, gpu_ctx).mat
        for k, dec in ((1, True), (10, True), (10, False), (40, True), (S, False)):
            fused = pb.score_topk(Xn, Gn, k, dec, ctx=gpu_ctx, **kw)
            assert_same(fused, pb.col_topk(full, k, dec, ctx=gpu_ctx), (name, k, dec))
            assert_same(fused, ref_topk(full, k, dec), (name, k, dec, "numpy"))
            idx, val = fused
            cols = np.arange(full.shape[1])[None, :]
            assert np.array_equal(val.view(np.int64), full[idx, cols].view(np.int64)), name


def test_column_tiles_beyond_device_memory(small_case, gpu_ctx, monkeypatch):
    Xn, Gn = small_case[:2]
    S = Gn.shape[1]
    for name, kw, _ in (SCORERS[0], SCORERS[2]):
        for k, dec in ((10, True), (64, False)):
            whole = pb.score_topk(Xn, Gn, k, dec, ctx=gpu_ctx, **kw)
            monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(S * 8 * 70))  # 64 columns per tile: 5 tiles
            tiled = pb.score_topk(Xn, Gn, k, dec, ctx=gpu_ctx, **kw)
            monkeypatch.delenv("PLAIDGPU_MAX_OUT_BYTES")
            assert_same(tiled, whole, (name, k, dec))


def test_several_contexts_and_ranks(small_case):
    from plaid_b200 import sharded
    from plaid_b200.api import _matrix_struct, _opts
    Xn, Gn, X, G, names = small_case
    N = Xn.shape[1]
    ctxs = [pb.Context(0) for _ in range(3)]
    for k, dec in ((10, True), (50, False)):
        one = pb.score_topk(Xn, Gn, k, dec, ctx=ctxs[0])
        for world in (2, 3):
            assert_same(pb.score_topk(Xn, Gn, k, dec, ctx=ctxs[:world]), one, (world, k, dec))
    # torch.distributed-style ranks (one thread and one context each)
    world, k = 3, 10
    one = pb.score_topk(Xn, Gn, k, ctx=ctxs[0])
    comms = sharded.ThreadComm.group(world)
    rowmap = pb.make_rowmap(names, names)
    res, errs = [None] * world, []

    def rank(r):
        try:
            c = ctxs[r]
            c.set_genesets(G)
            lo, hi = sharded.shard_columns(N, world, r)
            keep = []
            M = _matrix_struct(X[:, lo:hi], keep)
            o = _opts(c.lib, scorer=L.PLAID, stats_mean=1, normalize=1)
            res[r] = sharded.score_topk_shard(c, comms[r], M, rowmap, o, k, True, hi - lo)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)

    th = [threading.Thread(target=rank, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    got = (np.concatenate([r[0] for r in res], axis=1), np.concatenate([r[1] for r in res], axis=1))
    assert_same(got, one)


def test_real_set_count(gpu_ctx):
    """a C4-shaped collection: 30,000 synthetic sets over 20,000 genes, 4,096 cells"""
    P, N, S = 20000, 4096, 30000
    X = synth.sparse_x_numpy(P, N, seed=301)
    G = synth.genesets_numpy(P, S, seed=302)
    names = synth.gene_names(P)
    Xn, Gn = pb.NamedMatrix(X, names), pb.NamedMatrix(G, names)
    full = pb.plaid(Xn, Gn, ctx=gpu_ctx).mat
    wi, wv = ref_topk(full, 256, True)
    for k in (10, 256):  # the first k of a top-256 list are the top k
        assert_same(pb.score_topk(Xn, Gn, k, ctx=gpu_ctx), (wi[:k], wv[:k]), k)


def test_bad_arguments_are_rejected(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    S = Gn.shape[1]
    x = np.ones((3, 4))
    for k in (0, 4, 257):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.col_topk(x, k, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG, k
    for k in (0, S + 1, 257):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.score_topk(Xn, Gn, k, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG, k
    with pytest.raises(ValueError):
        pb.col_topk(np.ones(5), 1, ctx=gpu_ctx)
    with pytest.raises(ValueError):
        pb.col_topk(np.ones((2, 2, 2)), 1, ctx=gpu_ctx)
    lib = gpu_ctx.lib
    idx = np.empty((2, 4), dtype=np.int32)
    val = np.empty((2, 4))
    assert lib.plaidgpu_col_topk(gpu_ctx.h, None, 3, 4, 2, 1, L.HOST, idx.ctypes.data, val.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_col_topk(gpu_ctx.h, x.ctypes.data, 3, 4, 2, 1, L.HOST, None, val.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_col_topk(gpu_ctx.h, x.ctypes.data, 3, 4, 2, 1, L.HOST, idx.ctypes.data, None) == L.ERR_ARG
    # the fused calls: null X / idx / val, and the same context twice
    from plaid_b200.api import _matrix_struct, _opts
    gpu_ctx.set_genesets(Gn.mat)
    keep = []
    M = _matrix_struct(Xn.mat, keep)
    rowmap = pb.make_rowmap(Xn.rownames, Gn.rownames)
    o = _opts(lib, scorer=L.PLAID, stats_mean=1, normalize=1)
    N = M.N
    ti = np.empty((5, N), dtype=np.int32)
    tv = np.empty((5, N))
    args = (C.byref(M), rowmap.ctypes.data, C.byref(o), 5, 1)
    assert lib.plaidgpu_score_topk(gpu_ctx.h, None, rowmap.ctypes.data, C.byref(o), 5, 1, ti.ctypes.data,
                                   tv.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_topk(gpu_ctx.h, *args, None, tv.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_topk(gpu_ctx.h, *args, ti.ctypes.data, None) == L.ERR_ARG
    hs = (C.c_void_p * 2)(gpu_ctx.h, gpu_ctx.h)
    assert lib.plaidgpu_score_topk_multi(hs, 2, *args, ti.ctypes.data, tv.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_topk_multi(hs, 2, None, rowmap.ctypes.data, C.byref(o), 5, 1, ti.ctypes.data,
                                         tv.ctypes.data) == L.ERR_ARG
    # every multi-context entry point rejects the same context twice also with too few columns to split (N < 2n)
    M3 = _matrix_struct(Xn.mat[:, :3], keep)
    out3 = np.empty((S, 3), order="F")
    lab3 = np.zeros(3, dtype=np.int32)
    mom = np.empty((2, 2, S))
    args3 = (C.byref(M3), rowmap.ctypes.data, C.byref(o))
    assert lib.plaidgpu_score_multi(hs, 2, *args3, out3.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_group_stats_multi(hs, 2, *args3, lab3.ctypes.data, 2, mom.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_topk_multi(hs, 2, *args3, 5, 1, ti.ctypes.data, tv.ctypes.data) == L.ERR_ARG
    other = pb.Context(0)
    other.set_genesets(Gn.mat)
    hs = (C.c_void_p * 2)(gpu_ctx.h, other.h)
    og = _opts(lib, scorer=L.GSVA, tau=0.0, gsva_ecdf=1)
    assert lib.plaidgpu_score_topk_multi(hs, 2, C.byref(M), rowmap.ctypes.data, C.byref(og), 5, 1, ti.ctypes.data,
                                         tv.ctypes.data) == L.ERR_ARG
    # and a good call still works on this context afterwards
    assert lib.plaidgpu_score_topk(gpu_ctx.h, *args, ti.ctypes.data, tv.ctypes.data) == L.OK
    # after the fused calls, begin / compute / finish on the same context returns the scores themselves
    from plaid_b200 import sharded
    want = pb.plaid(Xn, Gn, ctx=other).mat
    lab = np.zeros(N, dtype=np.int32)
    mom = np.empty((2, 2, S))
    assert lib.plaidgpu_score_group_stats(gpu_ctx.h, *args[:3], lab.ctypes.data, 2, mom.ctypes.data) == L.OK
    assert lib.plaidgpu_score_topk(gpu_ctx.h, *args, ti.ctypes.data, tv.ctypes.data) == L.OK
    got = np.empty((S, N), order="F")
    sharded.score_shard(gpu_ctx, sharded.ThreadComm.group(1)[0], M, rowmap, o, got.ctypes.data, N)
    assert np.array_equal(got.view(np.int64), want.view(np.int64))
