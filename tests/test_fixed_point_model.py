"""An exact host model of the fixed-point route of plaid() (DESIGN §3.0), compared bit for bit.

k_tc_prep_csc / k_tc_prep_dense give every column j an exponent e_j = 30 - frexp(max |v|)[1] and round each entry to
q = rint(v * 2^e_j), half to even; k_tile_place / k_tail and k_tc_score add the integers exactly; the epilogue converts
the sum once to fp64, scales it by 2^-e_j (exact) and multiplies by inv_s = 1 / (1e-8 + n_s) (1 for stats = "sum").
Which entries set e_j: for sparse X the stored entries of every row that is in some set (block and tail rows alike),
for dense X every row, also rows in no set.  The route gives up, and the whole call takes the fp64 passes, when an
entry is not finite, when e_j is outside [-900, 900], or when a non-zero entry rounds to q = 0.

The normalised scores are the model's raw scores with the fix-up of k_fixup (fixup_value): each column's median
(exact order statistics; zeros dropped when the smallest score is 0) and mean(medians) from the host function
plaidgpu_combine_medians.

Routes: the sparse input has a tensor-core block (256 genes in ~390 sets each) and a tail pass with a partial last
tile (plan_info asserts both); the dense input runs the tensor-core block over every row.  Each boundary case is a
call of its own (one flag sends the whole call to fp64) and asserts the route the model predicts: bit-equal to the
model when it stays on fixed point, bit-equal to the exact_fp64 call when it falls back."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import plaid_b200 as pb
from plaid_b200 import _lib as L, api, synth

pytestmark = pytest.mark.gpu

NB, NT, NO = 256, 1744, 100  # block genes, tail genes, genes in no set
P, N, S = NB + NT + NO, 2500, 1100
TILE = 1056


@pytest.fixture(scope="module")
def ctx():
    c = pb.Context(0)
    yield c
    c.close()


def gene_sets(rng):
    """as in test_tail_atomic.py: 90 block genes per set (> 100,000 memberships), tail genes in < 32 sets each,
    the last NO genes in no set"""
    members = []
    for s in range(S):
        blk = (90 * s + np.arange(90)) % NB
        if s < 3:
            tl = np.arange(NB + 600 * s, min(NB + 600 * s + 1000, NB + NT))
        else:
            k = int(rng.integers(33, 100)) if s < 100 else int(rng.integers(0, 10))
            tl = rng.choice(np.arange(NB, NB + NT), size=k, replace=False)
        members.append(np.unique(np.concatenate([blk, tl])))
    gi = np.concatenate(members)
    gp = np.concatenate([[0], np.cumsum([m.size for m in members])])
    return sp.csc_matrix((np.ones(gi.size), gi, gp), shape=(P, S))


# special columns of the sparse input
C_TAILMAX, C_BLOCK_ONLY, C_TAIL_ONLY, C_EMPTY, C_HALF, C_NOSET = 10, 11, 12, 13, 14, 15


@pytest.fixture(scope="module")
def inputs():
    rng = np.random.default_rng(77)
    G = gene_sets(rng)
    X = np.zeros((P, N))
    lognorm = lambda *shape: rng.lognormal(0.0, 0.5, size=shape)  # noqa: E731
    X[:NB] = np.where(rng.random((NB, N)) < 0.3, lognorm(NB, N), 0.0)
    X[NB:NB + NT] = np.where(rng.random((NT, N)) < 0.05, lognorm(NT, N), 0.0)
    X[NB + NT:] = np.where(rng.random((NO, N)) < 0.05, lognorm(NO, N), 0.0)
    X[NB + 5:NB + 40] *= -1.0  # some negative addends
    X[:, C_TAILMAX] = 0.0
    X[:NB:3, C_TAILMAX] = lognorm(len(range(0, NB, 3)))
    X[NB + 7, C_TAILMAX] = 2.0 ** 16 * X[:NB, C_TAILMAX].max()  # the maximum is a tail entry, far above the block
    X[NB:, C_BLOCK_ONLY] = 0.0
    X[:NB, C_TAIL_ONLY] = 0.0
    X[:, C_EMPTY] = 0.0
    # v * 2^e_j = m + 0.5 exactly: e_j = 7 from the maximum 2^22 = 2^29 * 2^-7; q = rint(m + 0.5) rounds to even
    nz = np.flatnonzero(X[:NB + NT, C_HALF])
    X[nz, C_HALF] = (rng.integers(0, 1 << 20, size=nz.size) + 0.5) * 2.0 ** -7
    X[nz[0], C_HALF] = 2.0 ** 22
    # a row in no set holds by far the largest entry: it must not set e_j (sparse X)
    X[P - 1, C_NOSET] = 1e30
    # columns scaled by 2^k, k in [-800, 800]
    k = np.where(rng.random(N) < 0.5, rng.integers(-800, 801, size=N), 0)
    k[[C_TAILMAX, C_HALF, C_NOSET]] = 0
    X *= np.ldexp(1.0, k)[None, :]
    names = synth.gene_names(P)
    return X, G, names, k


def model_raw(X, G, stats_mean, dense):
    """(raw scores S x N, fallback predicted) of the fixed-point route; X dense array, zeros = not stored (sparse)"""
    deg = np.asarray((G != 0).sum(axis=1)).ravel()
    counted = np.ones(X.shape, bool) if dense else (X != 0) & (deg > 0)[:, None]
    V = np.where(counted, X, 0.0)
    if not np.isfinite(V).all():
        return None, True
    mx = np.abs(V).max(axis=0)
    e = np.where(mx > 0, 30 - np.frexp(mx)[1], 0)
    if (np.abs(e) > 900).any():
        return None, True
    Q = np.rint(V * np.ldexp(1.0, e)[None, :])  # exact scaling, half-to-even rounding
    if ((Q == 0) & (V != 0)).any():
        return None, True
    Qi = Q.astype(np.int64)
    Gi = sp.csc_matrix(G, dtype=np.int64)
    sums = np.asarray((Gi.T @ Qi))  # exact int64, |sum| < 2^51
    ns = np.asarray((G != 0).sum(axis=0)).ravel().astype(np.float64)
    inv = 1.0 / (1e-8 + ns) if stats_mean else np.ones(S)
    raw = (sums.astype(np.float64) * np.ldexp(1.0, -e)[None, :]) * inv[:, None]
    return raw, False


def _median(v):
    v = np.sort(v[~np.isnan(v)])
    n = v.size
    if n == 0:
        return 0.0
    a, b = v[(n - 1) // 2], v[n // 2]
    return a if n & 1 else (a + b) / 2.0


def model_normalised(raw, lib):
    smin = np.nanmin(raw)
    med_all = np.array([_median(raw[:, j]) for j in range(raw.shape[1])])
    med_nz = np.array([_median(np.where(raw[:, j] == 0, np.nan, raw[:, j])) for j in range(raw.shape[1])])
    scal = L.Scalars()
    assert lib.plaidgpu_combine_medians(-1, float(smin), med_all.ctypes.data, med_nz.ctypes.data, raw.shape[1],
                                        C.byref(scal)) == L.OK
    med = med_nz if scal.ignore_zero else med_all
    shift = (-med) + scal.med_mean  # fixup_value: alpha * (v + ((-med_j) + c)), alpha = 1
    return 1.0 * (raw + shift[None, :])


def _plaid(ctx, X, G, names, stats, normalize, dense, exact=False):
    old = api.EXACT_FP64
    api.EXACT_FP64 = exact
    try:
        Xm = np.asfortranarray(X) if dense else sp.csc_matrix(X)
        return pb.plaid(pb.NamedMatrix(Xm, names), pb.NamedMatrix(G, names), stats=stats, normalize=normalize,
                        ctx=ctx).mat
    finally:
        api.EXACT_FP64 = old


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def check(ctx, X, G, names, dense, stats="mean", normalize=False):
    """the call equals the model, or the exact_fp64 call when the model predicts a fallback; returns the prediction"""
    raw, fallback = model_raw(X, G, stats == "mean", dense)
    got = _plaid(ctx, X, G, names, stats, normalize, dense)
    info = ctx.plan_info()
    assert info["tc_rows"] > 0
    if not dense:  # the block is the NB high-degree genes, every other gene in a set is a tail row
        assert info["tc_rows"] == NB and info["tail_rows"] == NT and info["tail_tile_cells"] == TILE
    if fallback:
        assert bits_equal(got, _plaid(ctx, X, G, names, stats, normalize, dense, exact=True))
    else:
        want = model_normalised(raw, ctx.lib) if normalize else raw
        assert bits_equal(got, want), float(np.nanmax(np.abs(got - want)))
    return fallback


@pytest.mark.parametrize("stats", ["mean", "sum"])
@pytest.mark.parametrize("normalize", [False, True])
def test_sparse_matches_model(ctx, inputs, stats, normalize):
    X, G, names, _ = inputs
    assert sp.csc_matrix(G).nnz > 100_000
    assert not check(ctx, X, G, names, False, stats, normalize)
    # the cases the input is meant to reach
    raw, _ = model_raw(X, G, True, False)
    assert (raw[:, C_EMPTY] == 0).all()
    deg = np.asarray((G != 0).sum(axis=1)).ravel()
    top = int(np.argmax(np.where(deg > 0, np.abs(X[:, C_TAILMAX]), 0.0)))
    assert NB <= top < NB + NT and deg[top] > 0  # C_TAILMAX: e_j is set by a tail row
    assert np.abs(X[top, C_TAILMAX]) >= 2.0 ** 16 * np.abs(X[:NB, C_TAILMAX]).max()
    assert (X[:NB, C_TAIL_ONLY] == 0).all() and (X[NB:NB + NT, C_TAIL_ONLY] != 0).any()
    assert (X[NB:, C_BLOCK_ONLY] == 0).all() and (X[:NB, C_BLOCK_ONLY] != 0).any()
    assert np.argmax(np.abs(X[:, C_NOSET])) >= NB + NT  # the largest entry of C_NOSET is in a row in no set


@pytest.mark.parametrize("stats", ["mean", "sum"])
@pytest.mark.parametrize("normalize", [False, True])
def test_dense_matches_model(ctx, inputs, stats, normalize):
    """dense X: every row sets e_j, also a row in no set, whose entry here is 2^12 times the column's other entries"""
    X, G, names, _ = inputs
    rng = np.random.default_rng(3)
    D = rng.lognormal(0.0, 0.5, size=(P, 600)) * np.ldexp(1.0, rng.integers(-700, 700, size=600))[None, :]
    D[P - 1, :50] *= 2.0 ** 12
    assert not check(ctx, D, G, names, True, stats, normalize)


@pytest.mark.parametrize("case,e,fallback", [("exp", 900, False), ("exp", 901, True), ("exp", -900, False),
                                             ("exp", -901, True), ("half", 0, True), ("half_ulp", 0, False)])
@pytest.mark.parametrize("dense", [False, True])
def test_boundaries(ctx, inputs, case, e, fallback, dense):
    """e_j at the limits of [-900, 900], and the smallest entry at v * 2^e_j = 0.5 (rounds to 0: fallback) against
    0.5 + 1 ulp (rounds to 1): one call each, the route asserted through the model's prediction"""
    X, G, names, _ = inputs
    X = X[:, :64].copy() if not dense else np.random.default_rng(4).lognormal(0.0, 0.5, size=(P, 64))
    j = 20
    col = np.abs(X[:, j]) if dense else np.abs(np.where(np.asarray((G != 0).sum(axis=1)).ravel() > 0, X[:, j], 0.0))
    r = int(np.argmax(col))
    # column maximum f * 2^(30 - e) with f in [0.5, 1): e_j = e exactly.  The scaling can leave the maximum an ulp off
    # its target (below 2^29 would give e_j = 1), so the maximum is set exactly afterwards
    top = np.ldexp(0.75, 30 - e) if case == "exp" else 2.0 ** 29  # "half": e_j = 0
    X[:, j] *= top / col[r]
    X[r, j] = np.copysign(top, X[r, j])
    if case != "exp":
        small = int(np.flatnonzero((X[:, j] != 0) & (np.arange(P) != r) & (np.arange(P) < NB + NT))[0])
        X[small, j] = 0.5 if case == "half" else np.nextafter(0.5, 1.0)
    assert check(ctx, X, G, names, dense) == fallback


def test_fp64_route_scales_exactly(ctx, inputs):
    """exact_fp64: scaling column j by 2^k_j scales its raw scores by exactly 2^k_j"""
    X, G, names, k = inputs
    base = X * np.ldexp(1.0, -k)[None, :]
    a = _plaid(ctx, X, G, names, "mean", False, False, exact=True)
    b = _plaid(ctx, base, G, names, "mean", False, False, exact=True)
    assert bits_equal(a, b * np.ldexp(1.0, k)[None, :])

