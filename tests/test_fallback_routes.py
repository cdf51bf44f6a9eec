"""One fallback decision per call.  The fixed-point route (tensor-core block + integer tail sums, DESIGN §3.0) gives up
on a column with a non-finite entry, with an exponent e_j outside [-900, 900], or with a non-zero entry that rounds to
q = 0; the fp64 passes then score the context's columns.  A call decides this once for all its columns, so the result
does not depend on how the columns are split: every case below puts one such column in the LAST chunk, shard or
column tile only and asserts that the call equals the unsplit call and the exact_fp64 call bit for bit.

Routes reached (asserted through `_falls_back`, which runs plaidgpu_score_begin / _compute and reads Scalars.fp64:
plaid() falls back on the triggered column alone and not on the others; and through plan_info: a tensor-core block
and a tail pass):
  (a) pinned host output with early shipping: chunks leave as raw scores before the last chunk falls back, and
      plaidgpu_score_compute has to ship everything again;
  (b) plaidgpu_score_multi on 2 and 3 contexts: the shards that stayed on the fixed-point route score again in fp64;
  (c) column tiles of score_chunked (PLAIDGPU_MAX_OUT_BYTES): raw, normalised and score_to_file restart in fp64;
  (d) group stats, design stats and top-k on several contexts and on column tiles;
  (e) ThreadComm ranks through sharded.score_shard and score_*_shard."""
import ctypes as C
import os
import threading

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import plaid_b200 as pb
from plaid_b200 import _lib as L, api, sharded, synth
from plaid_b200.api import _matrix_struct, _opts

pytestmark = pytest.mark.gpu

P, N, S = 1500, 3200, 1800  # PLAIDGPU_TAIL_TILES=1: chunks of 1,056 columns, the last one [3168, 3200)
TRIGGERS = ("nan", "range", "flush")


@pytest.fixture(scope="module")
def base():
    X = sp.csc_matrix(synth.sparse_x_numpy(P, N, seed=97))
    G = sp.csc_matrix(synth.genesets_numpy(P, S, seed=98, size_cap=(5, 200)))
    names = synth.gene_names(P)
    return X, G, names


@pytest.fixture(scope="module")
def ctxs():
    cs = [pb.Context(0) for _ in range(3)]
    yield cs
    for c in cs:
        c.close()


def triggered(X, G, how, j=N - 1):
    """X with column j changed so that the fixed-point route must give up on it (and on nothing else)"""
    X = X.copy().tocsc()
    X.sort_indices()
    lo, hi = X.indptr[j], X.indptr[j + 1]
    rows = X.indices[lo:hi]
    member = np.asarray((G != 0).sum(axis=1)).ravel()[rows] > 0
    assert member.sum() >= 2
    a, b = lo + np.flatnonzero(member)[:2]  # two entries of rows in some set (block or tail: both set e_j)
    if how == "nan":
        X.data[a] = np.nan
    elif how == "range":  # e_j = 30 - frexp(max) > 900
        X.data[lo:hi] *= 2.0 ** -960
    else:  # one entry 2^-40 below the column maximum: q = rint(2^-40 * 2^30...) = 0
        X.data[b] = np.abs(X.data[lo:hi]).max() * 2.0 ** -40
    return X


def named(X, names):
    return pb.NamedMatrix(X, names)


def exact(f):
    old = api.EXACT_FP64
    api.EXACT_FP64 = True
    try:
        return f()
    finally:
        api.EXACT_FP64 = old


def _falls_back(ctx, X, G, names, **kw):
    """plaidgpu_score_begin / _compute on X; True when compute reports that the fixed-point route gave up"""
    ctx.set_genesets(G)
    keep = []
    M = _matrix_struct(X, keep)
    o = _opts(ctx.lib, **kw)
    o.out_location = L.HOST
    loc = L.Scalars()
    rowmap = pb.make_rowmap(names, names)
    ctx.check(ctx.lib.plaidgpu_score_begin(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), C.byref(loc)))
    ctx.check(ctx.lib.plaidgpu_score_compute(ctx.h, C.byref(loc), None))
    info = ctx.plan_info()
    assert info["tc_rows"] > 0 and info["tail_rows"] > 0
    return bool(loc.fp64)


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.int64) if a.dtype == np.float64 else a,
                                                 b.view(np.int64) if b.dtype == np.float64 else b)


def test_triggers_reach_the_fallback(ctxs, base):
    """each trigger sends its column (and only its column) off the fixed-point route; the untouched X stays on it"""
    X, G, names = base
    c = ctxs[0]
    plaid = dict(scorer=L.PLAID, stats_mean=1, normalize=1)
    assert not _falls_back(c, X, G, names, **plaid)
    for how in TRIGGERS:
        Xt = triggered(X, G, how)
        assert _falls_back(c, Xt[:, N - 1:], G, names, **plaid), how
        assert not _falls_back(c, Xt[:, :N - 1], G, names, **plaid), how
    # the rank scorers quantise transformed ranks: the NaN entry sends replaid.sing to the fp64 passes, while
    # replaid.ucell stays on fixed point
    Xt = triggered(X, G, "nan")
    for kw, falls in ((dict(scorer=L.UCELL, rmax=200.0, normalize=1), False), (dict(scorer=L.SING), True)):
        assert not _falls_back(c, X, G, names, **kw)
        assert _falls_back(c, Xt, G, names, **kw) == falls, kw


@pytest.mark.parametrize("how", TRIGGERS)
def test_late_chunk_after_early_shipping(ctxs, base, how, monkeypatch):
    """(a) pinned output, chunk 0 leaves early as raw scores, the last chunk falls back: the result equals the
    PLAIDGPU_NO_EARLY result and the exact_fp64 result, for plaid() normalised and replaid.sing (which fall back)
    and replaid.ucell (which stays on fixed point, where its rank sums are exact)."""
    X, G, names = base
    c = ctxs[0]
    Xn, Gn = named(triggered(X, G, how), names), named(G, names)
    monkeypatch.setenv("PLAIDGPU_TAIL_TILES", "1")
    calls = [lambda **kw: pb.plaid(Xn, Gn, ctx=c, **kw)]
    if how == "nan":  # replaid.sing falls back on this X, replaid.ucell does not (see above)
        calls += [lambda **kw: pb.replaid_ucell(Xn, Gn, rmax=200, ctx=c, **kw), lambda **kw: pb.replaid_sing(Xn, Gn, ctx=c, **kw)]
    for f in calls:
        monkeypatch.setenv("PLAIDGPU_NO_EARLY", "1")
        want = f().mat.copy()
        monkeypatch.delenv("PLAIDGPU_NO_EARLY")
        want64 = exact(lambda: f().mat.copy())
        monkeypatch.setenv("PLAIDGPU_EARLY_FRAC", "0.6")
        pinned = torch.empty(S * N, dtype=torch.float64).pin_memory()
        got = np.asarray(f(out=pinned.numpy().reshape((S, N), order="F")).mat)
        monkeypatch.delenv("PLAIDGPU_EARLY_FRAC")
        assert same(got, want) and same(got, want64)


@pytest.mark.parametrize("how", TRIGGERS)
def test_several_contexts(ctxs, base, how):
    """(b) plaidgpu_score_multi: the trigger is in the last shard; 2 and 3 contexts equal one context"""
    X, G, names = base
    Xn, Gn = named(triggered(X, G, how), names), named(G, names)
    for kw in (dict(), dict(normalize=False), dict(stats="sum", normalize=False)):
        one = pb.plaid(Xn, Gn, ctx=ctxs[0], **kw).mat
        assert same(one, exact(lambda: pb.plaid(Xn, Gn, ctx=ctxs[0], **kw).mat))
        for n in (2, 3):
            assert same(pb.plaid(Xn, Gn, ctx=ctxs[:n], **kw).mat, one), (kw, n)
    # the same protocol driven from Python (sharded.score_multi, one process, several contexts)
    Xt = triggered(X, G, how)
    spans = [sharded.shard_columns(N, 2, r) for r in range(2)]
    keep, outs, opts = [], [np.empty((S, hi - lo), order="F") for lo, hi in spans], []
    mats = [_matrix_struct(Xt[:, lo:hi], keep) for lo, hi in spans]
    for c in ctxs[:2]:
        c.set_genesets(G)
        opts.append(_opts(c.lib, scorer=L.PLAID, stats_mean=1, normalize=1, out_location=L.HOST))
    sharded.score_multi(ctxs[:2], mats, pb.make_rowmap(names, names), opts, [a.ctypes.data for a in outs],
                        [hi - lo for lo, hi in spans])
    assert same(np.concatenate(outs, axis=1), pb.plaid(Xn, Gn, ctx=ctxs[0]).mat)
    if how == "nan":
        one = pb.replaid_ucell(Xn, Gn, rmax=200, ctx=ctxs[0]).mat
        assert same(pb.replaid_ucell(Xn, Gn, rmax=200, ctx=ctxs[:2]).mat, one)


@pytest.mark.parametrize("how", TRIGGERS)
def test_column_tiles(ctxs, base, how, monkeypatch, tmp_path):
    """(c) score_chunked: the trigger is in the last of 7 column tiles; raw, normalised and score_to_file equal the
    untiled call"""
    X, G, names = base
    c = ctxs[0]
    Xn, Gn = named(triggered(X, G, how), names), named(G, names)
    raw = pb.plaid(Xn, Gn, ctx=c, normalize=False).mat
    norm = pb.plaid(Xn, Gn, ctx=c).mat
    monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(S * 8 * 500))  # 480 columns per tile
    assert same(pb.plaid(Xn, Gn, ctx=c, normalize=False).mat, raw)
    assert same(pb.plaid(Xn, Gn, ctx=c).mat, norm)
    path = os.path.join(str(tmp_path), "scores.npy")
    assert pb.score_to_file(Xn, Gn, path, ctx=c) == (S, N)
    assert same(np.load(path), norm)


@pytest.mark.parametrize("how", TRIGGERS)
def test_fused_targets(ctxs, base, how, monkeypatch):
    """(d) group stats, design stats and top-k on 2 contexts and on column tiles equal the same call in exact_fp64"""
    X, G, names = base
    Xn, Gn = named(triggered(X, G, how), names), named(G, names)
    rng = np.random.default_rng(5)
    labels = rng.integers(0, 4, size=N).astype(np.int32)
    B = np.column_stack([np.ones(N), rng.standard_normal(N)])
    calls = [lambda cx: pb.score_group_stats(Xn, Gn, labels, 4, ctx=cx),
             lambda cx: pb.score_design_stats(Xn, Gn, B, ctx=cx),
             lambda cx: pb.score_topk(Xn, Gn, 5, ctx=cx)]
    for tiled in (False, True):
        if tiled:
            monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(S * 8 * 500))
        cx = ctxs[0] if tiled else ctxs[:2]
        for f in calls:
            got, want = f(cx), exact(lambda: f(cx))
            if isinstance(got, tuple):
                assert same(got[0], want[0]) and same(got[1], want[1])
            else:
                assert same(got, want)


def _ranks(ctxs, world, X, G, names, run):
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
            res[r] = run(c, comms[r], M, rowmap, o, lo, hi)
        except Exception as e:  # pragma: no cover - reported below
            errs.append(e)

    th = [threading.Thread(target=rank, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    return res


@pytest.mark.parametrize("how", TRIGGERS)
def test_thread_ranks(ctxs, base, how):
    """(e) ThreadComm ranks: score_shard equals the one-context call; score_group_stats_shard,
    score_design_stats_shard and score_topk_shard equal the same ranks in exact_fp64"""
    X, G, names = base
    Xt = triggered(X, G, how)
    one = pb.plaid(named(Xt, names), named(G, names), ctx=ctxs[0]).mat

    def scores(c, comm, M, rowmap, o, lo, hi):
        out = np.empty((S, hi - lo), order="F")
        sharded.score_shard(c, comm, M, rowmap, o, out.ctypes.data, hi - lo)
        return out

    for world in (2, 3):
        got = np.concatenate(_ranks(ctxs, world, Xt, G, names, scores), axis=1)
        assert same(got, one), world
    rng = np.random.default_rng(6)
    labels = rng.integers(0, 3, size=N).astype(np.int32)
    B = np.column_stack([np.ones(N), rng.standard_normal(N)])
    fused = [lambda c, comm, M, rowmap, o, lo, hi: sharded.score_group_stats_shard(c, comm, M, rowmap, o, labels[lo:hi], 3, hi - lo),
             lambda c, comm, M, rowmap, o, lo, hi: sharded.score_design_stats_shard(c, comm, M, rowmap, o, B[lo:hi], hi - lo),
             lambda c, comm, M, rowmap, o, lo, hi: np.concatenate(
                 [a.astype(np.float64).ravel() for a in sharded.score_topk_shard(c, comm, M, rowmap, o, 5, True, hi - lo)])]
    for f in fused:
        got = _ranks(ctxs, 2, Xt, G, names, f)
        want = exact(lambda: _ranks(ctxs, 2, Xt, G, names, f))
        for a, b in zip(got, want):
            assert same(a, b)
