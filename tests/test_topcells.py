"""Per-row top k with cell indices (-m gpu): plaidgpu_row_topk against numpy's lexsort on every kind of row (ties,
signed zeros, infinities, NaN, constant and sorted rows) with one and many column chunks, the fused scoring call
(plaidgpu_score_row_topk) against scoring followed by the selection for seven scorers, column tiles beyond device
memory (ties across tile boundaries), several contexts and ThreadComm ranks, a C4-shaped set count, the fp64 fallback
in the last tile or shard, and rejected arguments.  Every comparison is exact: indices equal, values equal bit for
bit (NaN by isnan).  Every test runs twice (fixture `precision`, as in test_topk.py)."""
import ctypes as C
import threading

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import plaid_b200 as pb
from plaid_b200 import _lib as L, api, sharded, synth
from plaid_b200.api import _matrix_struct, _opts

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["tc", "fp64"])
def precision(request):
    old = api.EXACT_FP64
    api.EXACT_FP64 = request.param == "fp64"
    yield request.param
    api.EXACT_FP64 = old


def ref_row_topk(x, k, decreasing):
    """the first k entries of R's order(x[s, ], decreasing = decreasing) for every row (ties by column, NaN last)"""
    S, N = x.shape
    cols = np.arange(N)
    idx = np.empty((k, S), dtype=np.int64)
    val = np.empty((k, S))
    for s in range(S):
        v = x[s, :]
        o = np.lexsort((cols, -v if decreasing else v, np.isnan(v)))[:k]
        idx[:, s] = o
        val[:, s] = v[o]
    return idx, val


def assert_same(got, want, what=""):
    gi, gv = got
    wi, wv = want
    assert gi.shape == wi.shape and gv.shape == wv.shape, what
    assert np.array_equal(gi, wi), what
    nan = np.isnan(wv)
    assert np.array_equal(np.isnan(gv), nan), what
    assert np.array_equal(gv[~nan].view(np.int64), wv[~nan].view(np.int64)), what


def rows(rng, S, N, kind):
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
    if kind == "constant":  # with N >> k: ties across chunk boundaries must give the lowest columns
        return np.full((S, N), 2.25)
    if kind == "ascending":
        return np.repeat(np.arange(N, dtype=np.float64)[None, :], S, axis=0) + np.arange(S)[:, None]
    if kind == "descending":
        return np.repeat(-np.arange(N, dtype=np.float64)[None, :], S, axis=0) - np.arange(S)[:, None]
    raise ValueError(kind)


KINDS = ["normal", "ties", "zeros_inf", "some_nan", "all_nan", "constant", "ascending", "descending"]


# (1, 1), (7, 13): one chunk; (41, 257): four chunks; (9, 30000) and (70, 9000): 64 column chunks
@pytest.mark.parametrize("S,N", [(1, 1), (7, 13), (33, 70), (41, 257), (70, 9000), (9, 30000)])
def test_row_topk_matches_numpy(S, N, gpu_ctx):
    rng = np.random.default_rng(S * 7 + N)
    ks = sorted({k for k in (1, 31, 32, 33, 255, 256) if k <= N} | ({N} if N <= 256 else set()))
    for kind in KINDS:
        x = rows(rng, S, N, kind)
        xd = torch.from_numpy(np.asfortranarray(x).T.copy()).cuda()  # N x S row-major = S x N column-major
        for k in ks:
            for dec in (True, False):
                want = ref_row_topk(x, k, dec)
                assert_same(pb.row_topk(x, k, dec, ctx=gpu_ctx), want, (kind, k, dec, "host"))
                assert_same(pb.row_topk(pb.DeviceDense(xd, (S, N)), k, dec, ctx=gpu_ctx), want, (kind, k, dec, "device"))
    assert gpu_ctx.kernel_ms(2) >= 0.0


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
    N = Xn.shape[1]
    for name, kw, f in SCORERS:
        full = f(Xn, Gn, gpu_ctx).mat
        for k, dec in ((1, True), (10, True), (10, False), (40, True), (256, True), (N - 45, False)):
            fused = pb.score_row_topk(Xn, Gn, k, dec, ctx=gpu_ctx, **kw)
            assert_same(fused, pb.row_topk(full, k, dec, ctx=gpu_ctx), (name, k, dec))
            assert_same(fused, ref_row_topk(full, k, dec), (name, k, dec, "numpy"))
            idx, val = fused
            sets = np.arange(full.shape[0])[None, :]
            assert np.array_equal(val.view(np.int64), full[sets, idx].view(np.int64)), name


def tied_case(small_case):
    """every cell appears 30 times (columns j and j + 10 equal): all scores tie across tile and shard boundaries"""
    X, G, names = small_case[2:]
    Xr = sp.csc_matrix(X)[:, np.tile(np.arange(10), 30)]
    return pb.NamedMatrix(Xr, names), pb.NamedMatrix(G, names)


def test_column_tiles_beyond_device_memory(small_case, gpu_ctx, monkeypatch):
    S = small_case[1].shape[1]
    for Xn, Gn in (small_case[:2], tied_case(small_case)):
        for name, kw, f in (SCORERS[0], SCORERS[1], SCORERS[2]):  # normalised (two passes), raw, ucell
            full = f(Xn, Gn, gpu_ctx).mat
            for k, dec in ((10, True), (64, False), (100, True)):
                whole = pb.score_row_topk(Xn, Gn, k, dec, ctx=gpu_ctx, **kw)
                monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(S * 8 * 70))  # 64 columns per tile: 5 tiles
                tiled = pb.score_row_topk(Xn, Gn, k, dec, ctx=gpu_ctx, **kw)
                monkeypatch.delenv("PLAIDGPU_MAX_OUT_BYTES")
                assert_same(tiled, whole, (name, k, dec))
                assert_same(tiled, ref_row_topk(full, k, dec), (name, k, dec, "numpy"))


def _rank_results(ctxs, world, X, G, names, k, dec):
    N = X.shape[1]
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
            res[r] = sharded.score_row_topk_shard(c, comms[r], M, rowmap, o, k, dec, hi - lo, lo)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)

    th = [threading.Thread(target=rank, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    return res


def test_several_contexts_and_ranks(small_case):
    X, G, names = small_case[2:]
    ctxs = [pb.Context(0) for _ in range(3)]
    for Xn, Gn in (small_case[:2], tied_case(small_case)):
        for k, dec in ((10, True), (50, False), (150, True)):  # 150 > the 100 columns of a shard
            one = pb.score_row_topk(Xn, Gn, k, dec, ctx=ctxs[0])
            for world in (2, 3):  # 301 columns: ragged shards
                assert_same(pb.score_row_topk(Xn, Gn, k, dec, ctx=ctxs[:world]), one, (world, k, dec))
    for k, dec in ((10, True), (150, False)):
        one = pb.score_row_topk(small_case[0], small_case[1], k, dec, ctx=ctxs[0])
        for world in (2, 3):
            for got in _rank_results(ctxs, world, X, G, names, k, dec):  # every rank returns the whole result
                assert_same(got, one, (world, k, dec, "ranks"))


def test_real_set_count(gpu_ctx):
    """a C4-shaped collection: 30,000 synthetic sets over 20,000 genes, 600 cells"""
    P, N, S = 20000, 600, 30000
    X = synth.sparse_x_numpy(P, N, seed=301)
    G = synth.genesets_numpy(P, S, seed=302)
    names = synth.gene_names(P)
    Xn, Gn = pb.NamedMatrix(X, names), pb.NamedMatrix(G, names)
    full = pb.plaid(Xn, Gn, ctx=gpu_ctx).mat
    wi, wv = ref_row_topk(full, 256, True)
    for k in (10, 256):  # the first k of a top-256 list are the top k
        assert_same(pb.score_row_topk(Xn, Gn, k, ctx=gpu_ctx), (wi[:k], wv[:k]), k)


def triggered(X, G, how):
    """X with its last column changed so that the fixed-point route must give up on it (and on nothing else)"""
    X = sp.csc_matrix(X, copy=True)
    X.sort_indices()
    j = X.shape[1] - 1
    lo, hi = X.indptr[j], X.indptr[j + 1]
    member = np.asarray((G != 0).sum(axis=1)).ravel()[X.indices[lo:hi]] > 0
    a = lo + np.flatnonzero(member)[0]
    if how == "nan":
        X.data[a] = np.nan
    else:  # e_j = 30 - frexp(max) > 900
        X.data[lo:hi] *= 2.0 ** -960
    return X


@pytest.mark.parametrize("how", ["nan", "range"])
def test_fallback_in_the_last_tile_or_shard(small_case, how, monkeypatch):
    X, G, names = small_case[2:]
    S = G.shape[1]
    Xn, Gn = pb.NamedMatrix(triggered(X, G, how), names), pb.NamedMatrix(G, names)
    ctxs = [pb.Context(0) for _ in range(3)]

    def exact(f):
        old = api.EXACT_FP64
        api.EXACT_FP64 = True
        try:
            return f()
        finally:
            api.EXACT_FP64 = old

    for k, dec in ((10, True), (64, False)):
        want = exact(lambda: pb.score_row_topk(Xn, Gn, k, dec, ctx=ctxs[0]))
        assert_same(pb.score_row_topk(Xn, Gn, k, dec, ctx=ctxs[0]), want, (how, k, dec))
        for world in (2, 3):
            assert_same(pb.score_row_topk(Xn, Gn, k, dec, ctx=ctxs[:world]), want, (how, k, dec, world))
        monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(S * 8 * 70))
        assert_same(pb.score_row_topk(Xn, Gn, k, dec, ctx=ctxs[0]), want, (how, k, dec, "tiles"))
        monkeypatch.delenv("PLAIDGPU_MAX_OUT_BYTES")
        for got in _rank_results(ctxs, 2, triggered(X, G, how), G, names, k, dec):
            assert_same(got, want, (how, k, dec, "ranks"))


def test_bad_arguments_are_rejected(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    N = Xn.shape[1]
    x = np.ones((4, 3))
    for k in (0, 4, 257):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.row_topk(x, k, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG, k
    with pytest.raises(L.PlaidGpuError) as e:
        pb.row_topk(np.ones((2, 300)), 257, ctx=gpu_ctx)
    assert e.value.code == L.ERR_ARG
    for k in (0, 257):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.score_row_topk(Xn, Gn, k, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG, k
    with pytest.raises(ValueError):
        pb.row_topk(np.ones(5), 1, ctx=gpu_ctx)
    lib = gpu_ctx.lib
    idx = np.empty((2, 4), dtype=np.int64)
    val = np.empty((2, 4))
    assert lib.plaidgpu_row_topk(gpu_ctx.h, None, 4, 3, 2, 1, L.HOST, idx.ctypes.data, val.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_row_topk(gpu_ctx.h, x.ctypes.data, 4, 3, 2, 1, L.HOST, None, val.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_row_topk(gpu_ctx.h, x.ctypes.data, 4, 3, 2, 1, L.HOST, idx.ctypes.data, None) == L.ERR_ARG
    # the fused calls: k > N, null X / idx / val, the same context twice, gsva ecdf on several contexts
    gpu_ctx.set_genesets(Gn.mat)
    S = Gn.shape[1]
    keep = []
    M = _matrix_struct(Xn.mat, keep)
    rowmap = pb.make_rowmap(Xn.rownames, Gn.rownames)
    o = _opts(lib, scorer=L.PLAID, stats_mean=1, normalize=1)
    ti = np.empty((5, S), dtype=np.int64, order="F")
    tv = np.empty((5, S), order="F")
    M3 = _matrix_struct(Xn.mat[:, :3], keep)
    assert lib.plaidgpu_score_row_topk(gpu_ctx.h, C.byref(M3), rowmap.ctypes.data, C.byref(o), 4, 1, ti.ctypes.data,
                                       tv.ctypes.data) == L.ERR_ARG
    args = (C.byref(M), rowmap.ctypes.data, C.byref(o), 5, 1)
    assert lib.plaidgpu_score_row_topk(gpu_ctx.h, None, rowmap.ctypes.data, C.byref(o), 5, 1, ti.ctypes.data,
                                       tv.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_row_topk(gpu_ctx.h, *args, None, tv.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_row_topk(gpu_ctx.h, *args, ti.ctypes.data, None) == L.ERR_ARG
    hs = (C.c_void_p * 2)(gpu_ctx.h, gpu_ctx.h)
    assert lib.plaidgpu_score_row_topk_multi(hs, 2, *args, ti.ctypes.data, tv.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_row_topk_multi(hs, 2, C.byref(M3), rowmap.ctypes.data, C.byref(o), 2, 1, ti.ctypes.data,
                                             tv.ctypes.data) == L.ERR_ARG  # N < 2n
    assert lib.plaidgpu_score_row_topk_multi(hs, 2, None, rowmap.ctypes.data, C.byref(o), 5, 1, ti.ctypes.data,
                                             tv.ctypes.data) == L.ERR_ARG
    other = pb.Context(0)
    other.set_genesets(Gn.mat)
    hs = (C.c_void_p * 2)(gpu_ctx.h, other.h)
    assert lib.plaidgpu_score_row_topk_multi(hs, 2, C.byref(M), rowmap.ctypes.data, C.byref(o), N + 1, 1,
                                             ti.ctypes.data, tv.ctypes.data) == L.ERR_ARG
    og = _opts(lib, scorer=L.GSVA, tau=0.0, gsva_ecdf=1)
    assert lib.plaidgpu_score_row_topk_multi(hs, 2, C.byref(M), rowmap.ctypes.data, C.byref(og), 5, 1, ti.ctypes.data,
                                             tv.ctypes.data) == L.ERR_ARG
    # and a good call still works on this context afterwards, equal to the scores it selects from
    assert lib.plaidgpu_score_row_topk(gpu_ctx.h, *args, ti.ctypes.data, tv.ctypes.data) == L.OK
    assert_same((ti, tv), ref_row_topk(pb.plaid(Xn, Gn, ctx=other).mat, 5, True))
