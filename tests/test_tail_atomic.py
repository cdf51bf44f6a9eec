"""The integer tail pass (tail_kernels.cu, k_tail): shared-memory atomics into a u32 low word and a packed 16-bit
high counter per cell, with the rows of consecutive tail members packed into full 32-lane segments.

X holds integers below 2^30, so every column's fixed point holds its entries exactly and plaid(normalize = FALSE)
equals inv_s * sum_g x[g, j] computed on the host the same way (an exact integer sum, one conversion, one multiply
by 1 / (1e-8 + n_s)): the comparison is bit for bit.  The inputs are built so that the tensor-core block and the
tail pass both run and the tail sees
  * many members adding q close to 2^30 into the same cells (hundreds of carries per cell), and the same with
    negative q (borrows) and with both signs;
  * members without entries in a tile (empty rows inside a 32-member batch);
  * sets with more than 32 and more than 64 tail members;
  * rows longer than 32 and longer than 96 entries in a tile;
  * a partial last tile (2,500 cells = 1,056 + 1,056 + 388);
  * short rows that share cells, so that one packed segment holds several adds to one cell."""
import numpy as np
import pytest
import scipy.sparse as sp

import plaid_b200 as pb
from plaid_b200 import api, synth

pytestmark = pytest.mark.gpu

P, N, S = 2000, 2500, 1100
NB = 256  # block genes: each in ~387 sets (>= 32 = the degree threshold at this S)
TILE = 1056


@pytest.fixture(scope="module")
def ctx():
    return pb.Context(0)


@pytest.fixture(scope="module")
def inputs():
    rng = np.random.default_rng(2024)
    # ---- gene sets: 90 block genes per set, round robin (> 100,000 memberships in all: the tensor-core pass and the
    # tail pass need that many); tail members per the cases above
    members = []
    tail_pos = np.arange(NB, 1256)       # 1,000 genes with large positive entries in the hot cells
    tail_neg = np.arange(1256, P)        # 744 genes with large negative entries in the hot cells
    for s in range(S):
        blk = (90 * s + np.arange(90)) % NB
        if s == 0:
            tl = tail_pos                                # carries
        elif s == 1:
            tl = tail_neg                                # borrows
        elif s == 2:
            tl = np.arange(756, 1756)                    # both
        else:  # tail genes stay below 32 sets each
            k = int(rng.integers(33, 100)) if s < 100 else int(rng.integers(0, 10))
            tl = rng.choice(np.arange(NB, P), size=k, replace=False)
        members.append(np.unique(np.concatenate([blk, tl])))
    gi = np.concatenate(members)
    gp = np.concatenate([[0], np.cumsum([m.size for m in members])])
    G = sp.csc_matrix((np.ones(gi.size), gi, gp), shape=(P, S))

    # ---- X: integers, |x| < 2^30
    X = np.zeros((P, N), dtype=np.int64)
    X[:NB] = np.where(rng.random((NB, N)) < 0.3, rng.integers(1, 1000, size=(NB, N)), 0)
    hot = np.concatenate([np.arange(t, t + 20) for t in (0, TILE, 2 * TILE, N - 20)])
    big = (1 << 30) - 1 - rng.integers(0, 1 << 20, size=(P, hot.size))
    X[np.ix_(tail_pos, hot)] = big[tail_pos]
    X[np.ix_(tail_neg, hot)] = -big[tail_neg]
    extra = (rng.random((P - NB, N)) < 0.02) & (X[NB:] == 0)
    X[NB:] = np.where(extra, rng.integers(-1000, 1000, size=(P - NB, N)) | 1, X[NB:])
    X[NB:NB + 16] = np.where(rng.random((16, N)) < 0.6, rng.integers(1, 1 << 29, size=(16, N)), 0)  # > 96 per tile
    X[NB + 16:NB + 32] = np.where(rng.random((16, N)) < 0.06, rng.integers(-(1 << 29), 1 << 29, size=(16, N)) | 1,
                                  0)  # 32 - 96 per tile
    X[300:332] = 0
    X[300:332, [5, 6, 7, TILE + 5, 2 * TILE + 7]] = rng.integers(1, 1 << 29, size=(32, 5))  # short rows, shared cells
    empty = rng.choice(np.arange(NB + 32, P), size=300, replace=False)
    X[empty] = 0                                         # members with no entries anywhere
    X[np.ix_(empty[:100], hot[:20])] = 1 << 29           # ... or only in the first tile
    Xs = sp.csc_matrix(X.astype(np.float64))

    sums = (sp.csc_matrix(G.T.astype(np.int64)) @ sp.csc_matrix(X)).toarray()  # exact int64
    ns = np.asarray((G != 0).sum(axis=0)).ravel()
    want = sums.astype(np.float64) * (1.0 / (1e-8 + ns.astype(np.float64)))[:, None]
    names = synth.gene_names(P)
    return pb.NamedMatrix(Xs, names), pb.NamedMatrix(G, names), want, sums


def _plaid_raw(ctx, Xg, Gg, exact):
    old = api.EXACT_FP64
    api.EXACT_FP64 = exact
    try:
        return pb.plaid(Xg, Gg, normalize=False, ctx=ctx).mat
    finally:
        api.EXACT_FP64 = old


def test_tail_sums_bit_exact(ctx, inputs):
    Xg, Gg, want, sums = inputs
    got = _plaid_raw(ctx, Xg, Gg, False)
    info = ctx.plan_info()
    assert info["tc_rows"] > 0 and info["tail_rows"] > 0 and info["tail_tile_cells"] == TILE
    # the cases the inputs are meant to reach
    assert np.abs(sums[0]).max() > 1 << 38 and sums[1].min() < -(1 << 38)
    assert np.array_equal(got, want)


def test_fixed_point_matches_exact_fp64(ctx, inputs):
    Xg, Gg, want, _ = inputs
    a = _plaid_raw(ctx, Xg, Gg, False)
    b = _plaid_raw(ctx, Xg, Gg, True)
    scale = np.abs(b).max()
    assert np.abs(a - b).max() <= 2e-8 * scale


def test_rank_scorer_negative_terms_match_exact_fp64(ctx, inputs):
    """replaid.sing: column ranks shifted by the zero-group term, so tail addends of both signs on every column."""
    Xg, Gg, _, _ = inputs
    old = api.EXACT_FP64
    try:
        api.EXACT_FP64 = False
        a = pb.replaid_sing(Xg, Gg, ctx=ctx).mat
        assert ctx.plan_info()["tail_rows"] > 0
        api.EXACT_FP64 = True
        b = pb.replaid_sing(Xg, Gg, ctx=ctx).mat
    finally:
        api.EXACT_FP64 = old
    assert np.abs(a - b).max() <= 2e-8 * np.abs(b).max()
