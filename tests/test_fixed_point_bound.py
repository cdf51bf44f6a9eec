"""A per-score error bound for the scorers whose fixed-point scores the exact model of test_fixed_point_model.py cannot
reproduce bit for bit (their pow / exp2 / division / fma results may differ from numpy's by an ulp).

Each raw score (plaidgpu_score_compute into a device buffer, before the fix-up of plaidgpu_score_finish) is checked on
its own against ref = inv_s * sum_{g in s} y_gj [* c_j], summed in long double, where y = the oracle's transformed
values (the matrix oracle/plaid_oracle.py hands to plaid()) and c_j the column scale of replaid.scse:

  |gpu - ref| <= inv_s * (m_sj * 2^(-e_j - 1) + A ulp of (sum_s |y - f0| + |f0| * n_s)) [* c_j] + slack of c_j

  * e_j = 30 - frexp(max |y_gj - f0_j|)[1] over the entries the route quantises, f0_j = f(r0_j) the value of the
    column's zeros (subtracted before quantising on sparse input, added back as f0 * n_s in the epilogue);
  * m_sj = the number of quantised entries of set s in column j (rounding error <= 2^(-e_j - 1) each);
  * A = 8 on the all-integer routes (transform, subtraction, fma, multiplies: a few roundings per score); n_s + 8
    where an fp64 scatter pass adds the rest of the set;
  * replaid.scse: c_j = 100 / (sum_g |y_gj| + 1e-8), added in warp order on the device: (k_j + 4) ulp of |ref|.

Routes: sparse X with a tensor-core block and a tail pass (plan_info: tc_rows = 256, tail_rows > 0); dense X (every
row quantised); and the tensor-core block followed by the fp64 scatter pass (more than 65,535 non-block genes in
sets: no tail pass, TcParams.final = 0, tail_rows = 0).  Every case also asserts that the call stayed on the
fixed-point route (Scalars.fp64 = 0) and that the bound's first term is not vacuous (some scores err)."""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import plaid_b200 as pb
from oracle import plaid_oracle as O
from plaid_b200 import _lib as L, synth
from plaid_b200.api import _matrix_struct, _opts

pytestmark = pytest.mark.gpu

NB, NT = 256, 1744
P, N, S = NB + NT, 700, 1100
EPS = np.finfo(np.float64).eps
RMAX = 200.0


@pytest.fixture(scope="module")
def ctx():
    c = pb.Context(0)
    yield c
    c.close()


def gene_sets(p, rng):
    """90 block genes per set (in ~390 sets each: the tensor-core block), every other gene in one or two sets (below
    the block's degree threshold of 0.75 % of the sets)"""
    members = []
    for s in range(S):
        tl = NB + np.concatenate([np.arange(s, p - NB, S), [int(rng.integers(0, p - NB))]])
        members.append(np.unique(np.concatenate([(90 * s + np.arange(90)) % NB, tl])))
    gi = np.concatenate(members)
    gp = np.concatenate([[0], np.cumsum([m.size for m in members])])
    return sp.csc_matrix((np.ones(gi.size), gi, gp), shape=(p, S))


@pytest.fixture(scope="module")
def inputs():
    rng = np.random.default_rng(31)
    G = gene_sets(P, rng)
    X = np.zeros((P, N))
    X[:NB] = np.where(rng.random((NB, N)) < 0.3, rng.lognormal(0.5, 0.6, size=(NB, N)), 0.0)
    X[NB:] = np.where(rng.random((NT, N)) < 0.06, rng.lognormal(0.5, 0.6, size=(NT, N)), 0.0)
    D = rng.lognormal(0.5, 0.6, size=(P, 400))
    D[rng.random(D.shape) < 0.2] = 0.0  # zeros: replaid.scse's removeLog2 only transforms x > 0 of dense X
    return sp.csc_matrix(X), D, G, synth.gene_names(P)


def transformed(scorer, X, **kw):
    """the oracle's per-entry values y (dense P x N) and whether plaid() takes the set mean over them"""
    Xm = X
    dense_ranks = lambda r: r.toarray() if sp.issparse(r) else np.asarray(r, dtype=np.float64)  # noqa: E731
    if scorer == "sing":
        return dense_ranks(O.colranks(Xm, ties_method="min")) / Xm.shape[0] - 0.5, True
    if scorer == "ssgsea":
        r = dense_ranks(O.colranks(Xm, keep_zero=True, ties_method="average"))
        if kw["alpha"] != 0:
            r = r ** (1 + kw["alpha"])
        return r / np.nanmax(r) - 0.5, True
    if scorer == "ucell":
        r = dense_ranks(O.colranks(Xm, ties_method="average"))
        return np.minimum(np.max(r) - r, RMAX + 1), True
    if scorer == "aucell":
        r = dense_ranks(O.colranks(Xm, ties_method="average"))
        a = math.ceil(0.05 * Xm.shape[0])
        return 1.08 * np.maximum((r - (np.max(r) - a)) / a, 0), True
    if scorer == "scse":
        if sp.issparse(Xm):
            y = sp.csc_matrix(Xm, copy=True)
            if kw["removeLog2"]:
                y.data = np.exp2(y.data)
            return y.toarray(), False
        y = np.array(Xm, dtype=np.float64, copy=True)
        if kw["removeLog2"]:
            y[y > 0] = np.exp2(y[y > 0])
        return y, False
    if scorer == "gsva":
        zX = (Xm - O.row_means(Xm)[:, None]) / (1e-8 + O.mat_rowsds(Xm))[:, None]
        r = O.colranks(zX, signed=True, ties_method="average")
        return r / np.max(np.abs(r)), True
    raise ValueError(scorer)


OPTS = {"sing": dict(scorer=L.SING), "ucell": dict(scorer=L.UCELL, rmax=RMAX), "aucell": dict(scorer=L.AUCELL),
        "gsva": dict(scorer=L.GSVA)}


def raw_scores(ctx, Xm, G, names, scorer, **kw):
    """plaidgpu_score_begin / _compute into a device buffer: the raw scores before plaidgpu_score_finish"""
    if scorer == "ssgsea":
        o_kw = dict(scorer=L.SSGSEA, alpha=kw["alpha"])
    elif scorer == "scse":
        o_kw = dict(scorer=L.SCSE, remove_log2=1 if kw["removeLog2"] else 0, score_mean=0)
    else:
        o_kw = OPTS[scorer]
    ctx.set_genesets(G)
    keep = []
    M = _matrix_struct(Xm, keep)
    o = _opts(ctx.lib, **o_kw)
    o.out_location = L.DEVICE
    n = M.N
    buf = torch.empty(S * n, dtype=torch.float64, device="cuda:0")
    loc = L.Scalars()
    rowmap = pb.make_rowmap(names, names)
    ctx.check(ctx.lib.plaidgpu_score_begin(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), C.byref(loc)))
    ctx.check(ctx.lib.plaidgpu_score_compute(ctx.h, C.byref(loc), buf.data_ptr()))
    torch.cuda.synchronize()
    assert loc.fp64 == 0  # the fixed-point route ran to the end
    return buf.cpu().numpy().reshape((S, n), order="F")


def check_bound(got, y, mean, G, stored, quantised_rows, colscale=False, scatter=False):
    """the per-score bound of the module docstring; stored: entries of X that are stored (all of dense X)"""
    Gb = sp.csc_matrix(G, dtype=np.float64)
    ns = np.asarray(Gb.sum(axis=0)).ravel()
    inv = 1.0 / (1e-8 + ns) if mean else np.ones(S)
    zero = ~stored
    f0 = np.array([y[np.flatnonzero(zero[:, j])[0], j] if zero[:, j].any() else 0.0 for j in range(y.shape[1])])
    w = np.where(stored, y - f0[None, :], 0.0)  # what the route quantises (f0 * n_s comes back in the epilogue)
    q = stored & quantised_rows[:, None]
    mx = np.abs(np.where(q, w, 0.0)).max(axis=0)
    e = np.where(mx > 0, 30 - np.frexp(mx * (1 + 2.0 ** -50))[1], 0)  # an ulp up on the device cannot lower e_j
    m = np.asarray(Gb.T @ q.astype(np.float64))
    a = np.asarray(Gb.T @ np.abs(w)) + np.abs(f0)[None, :] * ns[:, None]
    ulps = (ns[:, None] + 8) if scatter else 8
    ref = np.asarray(Gb.T.astype(np.longdouble) @ y.astype(np.longdouble)) * inv[:, None].astype(np.longdouble)
    bound = inv[:, None] * (m * np.ldexp(0.5, -e)[None, :] + ulps * EPS * a)
    if colscale:
        cs = 100.0 / (np.abs(y).astype(np.longdouble).sum(axis=0) + 1e-8)
        ref = ref * cs[None, :]
        k = stored.sum(axis=0)
        bound = bound * cs.astype(np.float64)[None, :] + (k + 4)[None, :] * EPS * np.abs(ref.astype(np.float64))
    err = np.abs(got.astype(np.longdouble) - ref).astype(np.float64)
    worst = float(np.max(err / np.maximum(bound, 1e-300)))
    assert (err <= bound).all(), worst
    assert (err > 0).any()


CASES = [("sing", {}), ("ssgsea", dict(alpha=0.0)), ("ssgsea", dict(alpha=0.25)), ("ucell", {}), ("aucell", {}),
         ("scse", dict(removeLog2=True)), ("scse", dict(removeLog2=False))]


@pytest.mark.parametrize("scorer,kw", CASES, ids=[f"{s}-{kw}" for s, kw in CASES])
def test_sparse_block_and_tail(ctx, inputs, scorer, kw):
    X, _, G, names = inputs
    got = raw_scores(ctx, X, G, names, scorer, **kw)
    info = ctx.plan_info()
    assert info["tc_rows"] == NB and info["tail_rows"] == NT
    y, mean = transformed(scorer, X, **kw)
    stored = X.toarray() != 0
    if scorer == "ssgsea":  # keep.zero ranks: the zeros take rank 0, transformed to -0.5 like the GPU's f0
        assert np.all(y[~stored] == -0.5)
    check_bound(got, y, mean, G, stored, np.ones(P, bool), colscale=scorer == "scse")


@pytest.mark.parametrize("scorer,kw", CASES + [("gsva", {})], ids=[f"{s}-{kw}" for s, kw in CASES + [("gsva", {})]])
def test_dense(ctx, inputs, scorer, kw):
    _, D, G, names = inputs
    got = raw_scores(ctx, np.asfortranarray(D), G, names, scorer, **kw)
    assert ctx.plan_info()["tc_rows"] > 0
    y, mean = transformed(scorer, D, **kw)
    check_bound(got, y, mean, G, np.ones(D.shape, bool), np.ones(P, bool), colscale=scorer == "scse")


def test_block_then_fp64_scatter_route(ctx):
    """More than 65,535 non-block genes in sets (16-bit tail member ids): no tail pass, so the tensor-core block
    writes partial sums (TcParams.final = 0) and the fp64 scatter pass adds the other rows to them.  Only the stored
    block entries are quantised, and e_j is set by them alone.  plaid() and replaid.sing."""
    rng = np.random.default_rng(11)
    nt = 70_000
    p = NB + nt
    G = gene_sets(p, rng)
    n = 300
    X = sp.random(p, n, density=0.02, format="csc", random_state=np.random.RandomState(12),
                  data_rvs=lambda k: rng.lognormal(0.0, 1.0, size=k))
    X = sp.csc_matrix(X.toarray() * np.ldexp(1.0, rng.integers(-300, 300, size=n))[None, :])
    names = synth.gene_names(p)
    got = pb.plaid(pb.NamedMatrix(X, names), pb.NamedMatrix(G, names), normalize=False, ctx=ctx).mat
    info = ctx.plan_info()
    assert info["tc_rows"] == NB and info["tail_rows"] == 0
    blk = np.arange(p) < NB
    Xd = X.toarray()
    check_bound(got, Xd, True, G, Xd != 0, blk, scatter=True)
    got = raw_scores(ctx, X, G, names, "sing")
    assert ctx.plan_info()["tail_rows"] == 0
    y, mean = transformed("sing", X)
    check_bound(got, y, mean, G, Xd != 0, blk, scatter=True)
