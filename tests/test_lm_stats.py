"""The host statistics of plaid_lm (design_qr + lm_from_moments) without a GPU: moments computed by numpy from random
scores against numpy.linalg.lstsq with the textbook formulas, and against scipy.stats.linregress for D = [1, y]."""
import numpy as np
import pytest
from scipy import stats

from plaid_b200 import api


def _moments(x, U):
    return np.vstack([U.T @ x.T, x.sum(axis=1), (x * x).sum(axis=1)])


def _reference(x, D, Cm):
    """per set: lstsq coefficients, then c^T beta, sigma sqrt(c^T (D^T D)^-1 c), t and the two-sided p"""
    N, Q = D.shape
    beta, *_ = np.linalg.lstsq(D, x.T, rcond=None)
    res = x.T - D @ beta
    df = N - Q
    sigma = np.sqrt((res * res).sum(axis=0) / df)
    XtXi = np.linalg.inv(D.T @ D)
    out = []
    for c in Cm.T:
        est = c @ beta
        se = sigma * np.sqrt(c @ XtXi @ c)
        t = est / se
        out.append((est, se, t, 2 * stats.t.sf(np.abs(t), df)))
    return out


def _rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


@pytest.mark.parametrize("Q", [1, 3, 8])
def test_matches_lstsq(Q):
    rng = np.random.default_rng(Q)
    S, N = 40, 150
    D = np.column_stack([np.ones(N)] + [rng.normal(size=N) for _ in range(Q - 1)])
    x = rng.normal(size=(S, N)) + 2.0 + np.outer(rng.normal(size=S), D[:, -1])
    U, R = api.design_qr(D)
    assert np.allclose(U.T @ U, np.eye(Q)) and np.allclose(U @ R, D)
    Cm = rng.normal(size=(Q, 2))
    for contr in (None, Cm):
        tabs = api.lm_from_moments(_moments(x, U), R, N, contr)
        want = _reference(x, D, np.eye(Q) if contr is None else contr)
        assert len(tabs) == len(want)
        for tab, (est, se, t, p) in zip(tabs, want):
            assert tab.shape == (S, 6)
            assert _rel(tab[:, 0], est) < 1e-9
            assert _rel(tab[:, 1], se) < 1e-9
            assert _rel(tab[:, 3], t) < 1e-9
            assert _rel(tab[:, 4], p) < 1e-7
            assert np.allclose(tab[:, 2], x.mean(axis=1), rtol=1e-12)
            adj = np.minimum(1, np.minimum.accumulate((p * S / stats.rankdata(p, "ordinal"))[np.argsort(-p)]))
            assert np.allclose(np.sort(tab[:, 5])[::-1], adj, rtol=1e-12)


def test_simple_regression_matches_linregress():
    rng = np.random.default_rng(5)
    S, N = 12, 90
    y = rng.normal(size=N)
    x = rng.normal(size=(S, N)) + np.outer(rng.normal(size=S), y)
    D = np.column_stack([np.ones(N), y])
    U, R = api.design_qr(D)
    slope = api.lm_from_moments(_moments(x, U), R, N)[1]
    for s in range(S):
        lr = stats.linregress(y, x[s])
        assert abs(slope[s, 0] - lr.slope) < 1e-9 * abs(lr.slope)
        assert abs(slope[s, 1] - lr.stderr) < 1e-9 * lr.stderr
        assert abs(slope[s, 4] - lr.pvalue) < 1e-7 * max(lr.pvalue, 1e-300)


def test_no_residual_degrees_of_freedom_give_na():
    rng = np.random.default_rng(6)
    N = Q = 3
    D = np.column_stack([np.ones(N), np.arange(N), np.arange(N) ** 2.0])
    x = rng.normal(size=(5, N))
    U, R = api.design_qr(D)
    for tab in api.lm_from_moments(_moments(x, U), R, N):
        assert np.all(np.isfinite(tab[:, 0])) and np.all(np.isfinite(tab[:, 2]))  # the estimates stay
        assert np.all(np.isnan(tab[:, [1, 3, 4, 5]]))
    # a perfect fit (sigma = 0) also gives NA, and a NaN score makes only its own set NaN
    D = np.column_stack([np.ones(6), np.arange(6.0)])
    x = np.vstack([1.0 + 2.0 * np.arange(6.0), rng.normal(size=6), rng.normal(size=6)])
    x[2, 3] = np.nan
    U, R = api.design_qr(D)
    slope = api.lm_from_moments(_moments(x, U), R, 6)[1]
    assert abs(slope[0, 0] - 2.0) < 1e-12 and np.all(np.isnan(slope[0, [1, 3, 4]]))
    assert np.all(np.isfinite(slope[1]))
    assert np.all(np.isnan(slope[2]))


def test_bad_designs_are_rejected():
    N = 20
    one, y = np.ones(N), np.arange(N, dtype=float)
    for D in (np.column_stack([one, y, 2 * y - 1]),   # rank deficient
              np.column_stack([one, np.zeros(N)]),    # a zero column
              np.column_stack([one, y])[:1],          # fewer rows than columns
              np.column_stack([one, np.where(y == 3, np.nan, y)]),
              np.ones((N, 65)), np.ones((N, 0))):
        with pytest.raises(ValueError):
            api.design_qr(D)
    with pytest.raises(ValueError):
        api.lm_from_moments(np.zeros((3, 4)), np.eye(2), N, np.ones((3, 1)))  # contrasts need Q rows
