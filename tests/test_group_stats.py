"""Per-group moments for K sample groups (-m gpu): plaidgpu_group_stats against numpy, the fused scoring call
(plaidgpu_score_group_stats) against scoring + reducing, K = 2 against the two-group entry points, the column-tiled
route beyond device memory, several contexts, and plaid_test_groups against the oracle's plaid.test run once per
group.  Every test runs twice (fixture `precision`, as in test_gpu_parity.py)."""
import ctypes as C

import numpy as np
import pytest

import plaid_b200 as pb
from oracle import plaid_oracle as O
from plaid_b200 import _lib as L, synth

from conftest import rel_err

pytestmark = pytest.mark.gpu

TC_TOL = 2e-8


@pytest.fixture(autouse=True, params=["tc", "fp64"])
def precision(request):
    from plaid_b200 import api
    old = api.EXACT_FP64
    api.EXACT_FP64 = request.param == "fp64"
    yield request.param
    api.EXACT_FP64 = old


def tol(exact):
    """the tolerance of the all-fp64 path, or the fixed-point bound of the tensor-core pass"""
    from plaid_b200 import api
    return exact if api.EXACT_FP64 else max(exact, TC_TOL)


def _np_stats(x, labels, K):
    out = np.zeros((K, 2, x.shape[0]))
    for k in range(K):
        sel = x[:, labels == k]
        out[k, 0] = sel.sum(axis=1)
        out[k, 1] = (sel ** 2).sum(axis=1)
    return out


def _labels(rng, N, K, empty=None):
    lab = rng.integers(-1, K, size=N).astype(np.int32)
    if empty is not None:
        lab[lab == empty] = -1
    return lab


def test_group_stats_matches_numpy(gpu_ctx):
    rng = np.random.default_rng(7)
    for K in (1, 3, 17):
        for S, N in ((7, 1), (33, 130), (257, 4099)):  # odd S, ragged N (chunks of unequal width)
            lab = _labels(rng, N, K, empty=K - 1 if K > 1 else None)
            xi = rng.integers(-50, 51, size=(S, N)).astype(np.float64)
            got = pb.group_stats(xi, lab, K, ctx=gpu_ctx)
            assert got.shape == (K, 2, S)
            assert np.array_equal(got, _np_stats(xi, lab, K)), (K, S, N)
            if K > 1:
                assert not got[K - 1].any()  # the empty group
            xr = rng.normal(size=(S, N)) * 3.0 + 1.0
            assert rel_err(pb.group_stats(xr, lab, K, ctx=gpu_ctx), _np_stats(xr, lab, K)) < 1e-13, (K, S, N)


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
           ("sing", dict(scorer=L.SING, nrow_x=900), lambda Xn, Gn, c: pb.replaid_sing(Xn, Gn, ctx=c))]


def test_fused_equals_score_then_reduce(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    lab = _labels(np.random.default_rng(8), Xn.shape[1], 5, empty=3)
    for name, kw, f in SCORERS:
        fused = pb.score_group_stats(Xn, Gn, lab, 5, ctx=gpu_ctx, **kw)
        full = f(Xn, Gn, gpu_ctx).mat
        assert np.array_equal(fused, pb.group_stats(full, lab, 5, ctx=gpu_ctx)), name


def test_two_groups_equal_the_two_group_calls(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    y = (np.random.default_rng(9).random(Xn.shape[1]) < 0.4).astype(np.int32)
    for name, kw, f in SCORERS:
        got = pb.score_group_stats(Xn, Gn, y, 2, ctx=gpu_ctx, **kw)
        assert np.array_equal(got.reshape(4, -1), pb.score_group_moments(Xn, Gn, y, ctx=gpu_ctx, **kw)), name
        full = f(Xn, Gn, gpu_ctx).mat
        assert np.array_equal(pb.group_stats(full, y, 2, ctx=gpu_ctx).reshape(4, -1), pb.group_moments(full, y, ctx=gpu_ctx))


def test_column_tiles_beyond_device_memory(small_case, gpu_ctx, monkeypatch):
    Xn, Gn = small_case[:2]
    S, N = Gn.shape[1], Xn.shape[1]
    lab = _labels(np.random.default_rng(10), N, 6)
    for name, kw, _ in (SCORERS[0], SCORERS[2]):
        whole = pb.score_group_stats(Xn, Gn, lab, 6, ctx=gpu_ctx, **kw)
        monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(S * 8 * 70))  # 64 columns per tile: 5 tiles
        tiled = pb.score_group_stats(Xn, Gn, lab, 6, ctx=gpu_ctx, **kw)
        monkeypatch.delenv("PLAIDGPU_MAX_OUT_BYTES")
        assert rel_err(tiled, whole) < 1e-12, name


def test_several_contexts_and_ranks(small_case):
    from plaid_b200 import sharded
    from plaid_b200.api import _matrix_struct, _opts
    import threading
    Xn, Gn, X, G, names = small_case
    N, K = Xn.shape[1], 4
    lab = _labels(np.random.default_rng(11), N, K)
    ctxs = [pb.Context(0) for _ in range(3)]
    one = pb.score_group_stats(Xn, Gn, lab, K, ctx=ctxs[0])
    for world in (2, 3):
        got = pb.score_group_stats(Xn, Gn, lab, K, ctx=ctxs[:world])
        assert rel_err(got, one) < 1e-13, world
        assert np.array_equal(pb.score_group_stats(Xn, Gn, lab, K, ctx=ctxs[:world]), got), world
    # torch.distributed-style ranks (one thread and one context each)
    world = 3
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
            res[r] = sharded.score_group_stats_shard(c, comms[r], M, rowmap, o, lab[lo:hi], K, hi - lo)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)

    th = [threading.Thread(target=rank, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    for r in range(world):
        assert rel_err(res[r], one) < 1e-13
        assert np.array_equal(res[r], res[0])


def _check_against_oracle(X, xr, xc, G, gr, gc, groups, ctx, gsetX=None):
    keep = np.array([g is not None and g == g for g in groups])
    kept = np.flatnonzero(keep)
    got = pb.plaid_test_groups(pb.NamedMatrix(X, xr, xc), groups, pb.NamedMatrix(G, gr, gc),
                               None if gsetX is None else pb.NamedMatrix(gsetX), ctx=ctx)
    levels = sorted(set(g for g, k in zip(groups, keep) if k))
    assert list(got) == levels
    Xk = X[:, kept]
    for lev in levels:
        y = np.array([groups[j] == lev for j in kept], dtype=int)
        og = None if gsetX is None else O.Named(gsetX[:, kept])
        want = O.plaid_test(O.Named(Xk, xr, [xc[j] for j in kept] if xc else None), y, O.Named(G, gr, gc), og)
        tab, cols, rows = got[lev]
        assert cols == want[1] and sorted(rows) == sorted(want[2])
        go, wo = np.argsort(rows), np.argsort(want[2])
        assert rel_err(tab[go], want[0][wo]) < tol(1e-8), lev


def test_plaid_test_groups_matches_oracle(fixture_mats, golden, gpu_ctx):
    X, xr, xc, G, gr, gc = fixture_mats
    celltype = [str(s) for s in golden["celltype"]]
    _check_against_oracle(X, xr, xc, G, gr, gc, celltype, gpu_ctx)
    # K = 5 with a one-cell group and cells left out (None / NaN)
    P, N, S = 700, 90, 60
    Xs = synth.sparse_x_numpy(P, N, seed=211, density=0.3)
    Gs = synth.genesets_numpy(P, S, seed=212, size_cap=(5, 100))
    names, sets = synth.gene_names(P), synth.set_names(S)
    rng = np.random.default_rng(12)
    groups = [int(v) for v in rng.integers(0, 4, size=N)]
    groups[5] = 9                       # the only cell of group 9
    for j in (1, 17, 40):
        groups[j] = None
    groups[60] = float("nan")
    _check_against_oracle(Xs, names, None, Gs, names, sets, groups, gpu_ctx)
    gsetX = pb.plaid(pb.NamedMatrix(Xs, names), pb.NamedMatrix(Gs, names), ctx=gpu_ctx).mat
    _check_against_oracle(Xs, names, None, Gs, names, sets, groups, gpu_ctx, gsetX=gsetX)


def test_bad_labels_are_rejected(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    x = np.ones((3, 4))
    for lab, K in (([0, 1, 2, 0], 2), ([0, -2, 1, 0], 2), ([0, 0, 0, 0], 0)):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.group_stats(x, lab, K, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG
    N = Xn.shape[1]
    for lab, K in ((np.full(N, 3), 3), (np.full(N, -2), 3), (np.zeros(N), 0)):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.score_group_stats(Xn, Gn, lab, K, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG
    with pytest.raises(ValueError):
        pb.group_stats(x, [0, 1, 0], 2, ctx=gpu_ctx)
    with pytest.raises(ValueError):
        pb.score_group_stats(Xn, Gn, np.zeros(N - 1), 2, ctx=gpu_ctx)
    lib = gpu_ctx.lib
    out = np.empty(12)
    assert lib.plaidgpu_group_stats(gpu_ctx.h, x.ctypes.data, 3, 4, None, 2, L.HOST, out.ctypes.data) == L.ERR_ARG
    lab = np.zeros(4, dtype=np.int32)
    assert lib.plaidgpu_group_stats(gpu_ctx.h, x.ctypes.data, 3, 4, lab.ctypes.data, 2, L.HOST, None) == L.ERR_ARG
    hs = (C.c_void_p * 2)(gpu_ctx.h, gpu_ctx.h)
    assert lib.plaidgpu_score_group_stats_multi(hs, 2, None, None, None, None, 2, None) == L.ERR_ARG
