"""Per-set products with a dense design (-m gpu): plaidgpu_design_stats against numpy, the fused scoring call
(plaidgpu_score_design_stats) against scoring + reducing, a one-hot design against the group sums, the column-tiled
route beyond device memory, several contexts and ranks, plaid_lm against least squares on the downloaded scores, and
the rejected arguments.  Every test runs twice (fixture `precision`, as in test_group_stats.py)."""
import ctypes as C
import threading

import numpy as np
import pytest
import torch

import plaid_b200 as pb
from plaid_b200 import _lib as L, synth

from conftest import rel_err
from test_group_stats import SCORERS

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["tc", "fp64"])
def precision(request):
    from plaid_b200 import api
    old = api.EXACT_FP64
    api.EXACT_FP64 = request.param == "fp64"
    yield request.param
    api.EXACT_FP64 = old


def _np_design(x, B):
    """the moments in extended precision: (Q + 2, S)"""
    xl, Bl = x.astype(np.longdouble), B.astype(np.longdouble)
    return np.vstack([(xl @ Bl).T, xl.sum(axis=1), (xl * xl).sum(axis=1)]).astype(np.float64)


def test_design_stats_matches_numpy(gpu_ctx):
    rng = np.random.default_rng(21)
    for Q in (1, 3, 32, 33, 64):
        for S, N in ((7, 1), (33, 130), (257, 4099)):
            xi = rng.integers(-50, 51, size=(S, N)).astype(np.float64)
            Bi = rng.integers(-5, 6, size=(N, Q)).astype(np.float64)
            xr = rng.normal(size=(S, N)) * 3.0 + 1.0
            Br = rng.normal(size=(N, Q)) + 0.5
            for x, B, exact in ((xi, Bi, True), (xr, Br, False)):
                want = _np_design(x, B)
                xd = torch.from_numpy(np.asfortranarray(x).T.copy()).cuda()  # N x S row-major = S x N column-major
                for where, arg in (("host", x), ("device", pb.DeviceDense(xd, (S, N)))):
                    got = pb.design_stats(arg, B, ctx=gpu_ctx)
                    assert got.shape == (Q + 2, S)
                    if exact:
                        assert np.array_equal(got, want), (Q, S, N, where)
                    else:
                        assert rel_err(got, want) < 1e-13, (Q, S, N, where)
    assert gpu_ctx.kernel_ms(2) >= 0.0


@pytest.fixture(scope="module")
def small_case():
    P, N, S = 900, 301, 131
    X = synth.sparse_x_numpy(P, N, seed=201, density=0.3)
    G = synth.genesets_numpy(P, S, seed=202, size_cap=(5, 120))
    names = synth.gene_names(P)
    return pb.NamedMatrix(X, names), pb.NamedMatrix(G, names, synth.set_names(S)), X, G, names


def _basis(rng, N, Q):
    D = np.column_stack([np.ones(N)] + [rng.normal(size=N) for _ in range(Q - 1)])
    return pb.design_qr(D)[0]


def test_fused_equals_score_then_reduce(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    rng = np.random.default_rng(22)
    for Q in (2, 40):
        U = _basis(rng, Xn.shape[1], Q)
        for name, kw, f in SCORERS:
            fused = pb.score_design_stats(Xn, Gn, U, ctx=gpu_ctx, **kw)
            full = f(Xn, Gn, gpu_ctx).mat
            assert np.array_equal(fused, pb.design_stats(full, U, ctx=gpu_ctx)), (name, Q)


def test_onehot_design_equals_group_sums(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    N, K = Xn.shape[1], 5
    lab = np.random.default_rng(23).integers(0, K, size=N).astype(np.int32)
    onehot = np.zeros((N, K))
    onehot[np.arange(N), lab] = 1.0
    for name, kw, _ in SCORERS:
        got = pb.score_design_stats(Xn, Gn, onehot, ctx=gpu_ctx, **kw)
        gs = pb.score_group_stats(Xn, Gn, lab, K, ctx=gpu_ctx, **kw)
        assert rel_err(got[:K], gs[:, 0]) < 1e-13, name
        assert rel_err(got[K], gs[:, 0].sum(axis=0)) < 1e-13, name
        assert rel_err(got[K + 1], gs[:, 1].sum(axis=0)) < 1e-13, name


def test_column_tiles_beyond_device_memory(small_case, gpu_ctx, monkeypatch):
    Xn, Gn = small_case[:2]
    S, N = Gn.shape[1], Xn.shape[1]
    U = _basis(np.random.default_rng(24), N, 6)
    for name, kw, _ in (SCORERS[0], SCORERS[2]):
        whole = pb.score_design_stats(Xn, Gn, U, ctx=gpu_ctx, **kw)
        monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(S * 8 * 70))  # 64 columns per tile: 5 tiles
        tiled = pb.score_design_stats(Xn, Gn, U, ctx=gpu_ctx, **kw)
        monkeypatch.delenv("PLAIDGPU_MAX_OUT_BYTES")
        assert rel_err(tiled, whole) < 1e-12, name


def test_several_contexts_and_ranks(small_case):
    from plaid_b200 import sharded
    from plaid_b200.api import _matrix_struct, _opts
    Xn, Gn, X, G, names = small_case
    N = Xn.shape[1]
    U = _basis(np.random.default_rng(25), N, 4)
    ctxs = [pb.Context(0) for _ in range(3)]
    one = pb.score_design_stats(Xn, Gn, U, ctx=ctxs[0])
    for world in (2, 3):
        got = pb.score_design_stats(Xn, Gn, U, ctx=ctxs[:world])
        assert rel_err(got, one) < 1e-13, world
        assert np.array_equal(pb.score_design_stats(Xn, Gn, U, ctx=ctxs[:world]), got), world
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
            res[r] = sharded.score_design_stats_shard(c, comms[r], M, rowmap, o, U[lo:hi], hi - lo)
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


def _lstsq_stats(x, D, Cm):
    from scipy import stats
    N, Q = D.shape
    beta, *_ = np.linalg.lstsq(D, x.T, rcond=None)
    res = x.T - D @ beta
    sigma = np.sqrt((res * res).sum(axis=0) / (N - Q))
    XtXi = np.linalg.inv(D.T @ D)
    out = []
    for c in Cm.T:
        est = c @ beta
        se = sigma * np.sqrt(c @ XtXi @ c)
        out.append((est, se, est / se, 2 * stats.t.sf(np.abs(est / se), N - Q)))
    return out


def _rel(a, b):
    return float(np.max(np.abs(a - b) / np.abs(b)))


def test_plaid_lm_matches_lstsq(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    N = Xn.shape[1]
    rng = np.random.default_rng(26)
    gsetX = pb.plaid(Xn, Gn, ctx=gpu_ctx).mat
    y = rng.normal(size=N)
    grp = rng.integers(0, 3, size=N)
    batch = (rng.random(N) < 0.5).astype(float)
    D2 = np.column_stack([np.ones(N), y])
    D3 = np.column_stack([np.ones(N), grp == 1, grp == 2, batch]).astype(float)
    Cm = np.array([[0, 1, 0, 0], [0, 0, 1, 0], [0, -1, 1, 0]], dtype=float).T  # g1 - g0, g2 - g0, g2 - g1
    for D, contr, names in ((D2, None, ["intercept", "y"]), (D3, Cm, ["g1", "g2", "g2-g1"])):
        want = _lstsq_stats(gsetX, D, np.eye(D.shape[1]) if contr is None else contr)
        design = pb.NamedMatrix(D, None, ["intercept", "y"] if contr is None else None)
        contrasts = None if contr is None else pb.NamedMatrix(contr, None, names)
        for src in ("fused", "gsetX"):
            got = pb.plaid_lm(Xn, Gn, design, contrasts, gsetX=None if src == "fused" else pb.NamedMatrix(gsetX),
                              ctx=gpu_ctx)
            assert list(got) == names
            for name, (est, se, t, p) in zip(names, want):
                tab, cols, rows = got[name]
                assert cols == ["logFC", "SE", "AveExpr", "t", "P.Value", "adj.P.Val"]
                assert rows == list(Gn.colnames)
                assert rel_err(tab[:, 0], est) < 1e-9, (name, src)
                assert _rel(tab[:, 1], se) < 1e-9, (name, src)
                assert rel_err(tab[:, 3], t) < 1e-9, (name, src)
                assert np.allclose(tab[:, 4], p, rtol=1e-6, atol=1e-300)
                assert np.allclose(tab[:, 2], gsetX.mean(axis=1), rtol=1e-12)
    tab, cols, rows = pb.plaid_lm(Xn, Gn, D2, sort_by="P.Value", ctx=gpu_ctx)["coef2"]
    assert np.all(np.diff(tab[:, 4]) >= 0) and sorted(rows) == sorted(Gn.colnames)


def test_plaid_lm_two_groups_equal_plaid_test(small_case, gpu_ctx):
    Xn, Gn = small_case[:2]
    N = Xn.shape[1]
    y = (np.random.default_rng(27).random(N) < 0.4).astype(int)
    got = pb.plaid_lm(Xn, Gn, np.column_stack([np.ones(N), y]), ctx=gpu_ctx)["coef2"]
    want = pb.plaid_test(Xn, y, Gn, tests=("lm",), sort_by="none", ctx=gpu_ctx)
    assert got[2] == want[2]
    assert rel_err(got[0][:, 0], want[0][:, 0]) < 1e-10


def test_bad_arguments_are_rejected(small_case, gpu_ctx):
    from plaid_b200.api import _matrix_struct, _opts
    Xn, Gn = small_case[:2]
    x = np.ones((3, 4))
    for B in (np.ones((4, 0)), np.ones((4, 65)), np.array([[1.0], [np.nan], [0.0], [1.0]]),
              np.array([[1.0], [np.inf], [0.0], [1.0]])):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.design_stats(x, B, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG
    N = Xn.shape[1]
    for B in (np.ones((N, 0)), np.ones((N, 65)), np.where(np.arange(N) == 7, np.nan, 1.0)):
        with pytest.raises(L.PlaidGpuError) as e:
            pb.score_design_stats(Xn, Gn, B, ctx=gpu_ctx)
        assert e.value.code == L.ERR_ARG
    with pytest.raises(ValueError):
        pb.design_stats(x, np.ones((3, 1)), ctx=gpu_ctx)
    with pytest.raises(ValueError):
        pb.plaid_lm(Xn, Gn, np.ones((N - 1, 1)), ctx=gpu_ctx)
    with pytest.raises(ValueError):  # rank deficient
        pb.plaid_lm(Xn, Gn, np.column_stack([np.ones(N), np.arange(N), 2.0 * np.arange(N) + 1]), ctx=gpu_ctx)
    with pytest.raises(ValueError):
        pb.plaid_lm(Xn, Gn, np.where(np.arange(N) == 3, np.nan, 1.0), ctx=gpu_ctx)
    lib = gpu_ctx.lib
    S = Gn.shape[1]
    B = np.ones((4, 2), order="F")
    out = np.empty(4 * 3)
    assert lib.plaidgpu_design_stats(gpu_ctx.h, None, 3, 4, B.ctypes.data, 2, L.HOST, out.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_design_stats(gpu_ctx.h, x.ctypes.data, 3, 4, None, 2, L.HOST, out.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_design_stats(gpu_ctx.h, x.ctypes.data, 3, 4, B.ctypes.data, 2, L.HOST, None) == L.ERR_ARG
    gpu_ctx.set_genesets(Gn.mat)
    keep = []
    M = _matrix_struct(Xn.mat, keep)
    rowmap = pb.make_rowmap(Xn.rownames, Gn.rownames)
    o = _opts(lib, scorer=L.PLAID, stats_mean=1, normalize=1)
    U = np.asfortranarray(_basis(np.random.default_rng(28), N, 2))
    mom = np.empty((4, S))
    args = (C.byref(M), rowmap.ctypes.data, C.byref(o))
    assert lib.plaidgpu_score_design_stats(gpu_ctx.h, None, rowmap.ctypes.data, C.byref(o), U.ctypes.data, 2,
                                           mom.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_design_stats(gpu_ctx.h, *args, None, 2, mom.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_design_stats(gpu_ctx.h, *args, U.ctypes.data, 2, None) == L.ERR_ARG
    # the same context twice, also with too few columns to split (N < 2n)
    hs = (C.c_void_p * 2)(gpu_ctx.h, gpu_ctx.h)
    assert lib.plaidgpu_score_design_stats_multi(hs, 2, *args, U.ctypes.data, 2, mom.ctypes.data) == L.ERR_ARG
    M3 = _matrix_struct(Xn.mat[:, :3], keep)
    assert lib.plaidgpu_score_design_stats_multi(hs, 2, C.byref(M3), rowmap.ctypes.data, C.byref(o), U.ctypes.data,
                                                 2, mom.ctypes.data) == L.ERR_ARG
    assert lib.plaidgpu_score_design_stats_multi(hs, 2, None, rowmap.ctypes.data, C.byref(o), U.ctypes.data, 2,
                                                 mom.ctypes.data) == L.ERR_ARG
    other = pb.Context(0)
    other.set_genesets(Gn.mat)
    hs = (C.c_void_p * 2)(gpu_ctx.h, other.h)
    og = _opts(lib, scorer=L.GSVA, tau=0.0, gsva_ecdf=1)
    assert lib.plaidgpu_score_design_stats_multi(hs, 2, C.byref(M), rowmap.ctypes.data, C.byref(og), U.ctypes.data,
                                                 2, mom.ctypes.data) == L.ERR_ARG
    # and a good call still works on this context afterwards
    assert lib.plaidgpu_score_design_stats(gpu_ctx.h, *args, U.ctypes.data, 2, mom.ctypes.data) == L.OK
