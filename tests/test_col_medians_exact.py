"""Per-column medians of the statistics pass, bit for bit, on every route (plaid_b200/csrc/stats_kernels.cu).

The medians are exact order statistics (DESIGN §3.3), so nothing here has a tolerance: every median, column
minimum and normalised value is compared bit for bit with a numpy model (NaN by isnan, -0 equal to +0).  Three
kernels compute the medians and two apply them:
  * k_colstats            three-pass radix select: S < 4096, and every column a one-pass kernel rejected;
  * k_colstats_one<NZ>    one median, S >= 4096 (ignore.zero given, every scoring call);
  * k_colstats_fast<1,1>  both medians, S >= 4096 (ignore.zero = NULL, the column-tiled scoring route);
  * k_fixup_flat / k_fixup  out = x + (c - med): even S >= 4096 / everything else.
A one-pass kernel that rejects a column hands it to k_colstats, so a wrong reject only costs time and a wrong
accept gives a wrong median: ROUTES says which kernel must accept which kind of column, and test_route_table
checks it through PLAIDGPU_TRACE_COLSTATS.

Each kind of column is a generator in CATALOGUE; its comment names the branch it targets, and it asserts on the
CPU what it can check without the kernel (where the median ranks fall, which rows are sampled, which residue
classes hold what).  `route_model` restates the accept / reject decision of the two one-pass kernels from their
sampling, bracket and capacity rules, so the route table is rehearsed on the CPU as well
(test_catalogue_self_checks needs no GPU).
"""
import ctypes as C
import re

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import plaid_oracle as O

pytestmark = pytest.mark.gpu

SHAPES = (4095, 4096, 4097, 6143, 30000, 70000)
S_ROUTE = 30000      # one launch per kind for the route table
S_CAP = 32768        # the capacity kinds: 128 rows per thread, sampled rows are the rows = 0 (mod 32)
NT, SAMP = 256, 1024  # column CTA threads; sample points of the one-pass kernels
TCAP, OVF, WCAP = 20, 512, 416


# ---- numpy model of the quantities the kernels work with ----------------------------------------------------
def ranks(n):
    """0-based ranks of the two middles of n sorted values"""
    return (n - 1) // 2, n // 2


def sample_rows(S):
    return (np.arange(SAMP, dtype=np.int64) * S) // SAMP


def dkey(v):
    """key_of (common.cuh): order-preserving uint64 of a double, -0 mapped to +0"""
    v = np.where(v == 0.0, 0.0, np.asarray(v, dtype=np.float64))
    b = v.view(np.uint64)
    return np.where(b >> np.uint64(63), ~b, b | np.uint64(1 << 63))


def fkey(f):
    b = np.asarray(f, dtype=np.float32).view(np.uint32)
    return np.where(b >> np.uint32(31), ~b, b | np.uint32(1 << 31))


def fval(k):
    k = np.uint32(k)
    return np.array(k & np.uint32(0x7FFFFFFF) if k >> np.uint32(31) else ~k, dtype=np.uint32).view(np.float32)[()]


def bracket_ranks(m):
    """sample ranks a, b of the bracket (2.5 sigma of a binomial(m, 1/2) rank); None = open end"""
    if m < 48:
        return None, None
    mid, delta = 0.5 * (m - 1), 1.25 * np.sqrt(m) + 2.0
    a, b = int(np.floor(mid - delta)), int(np.ceil(mid + delta))
    return (a if a >= 0 else None), (b if b <= m - 1 else None)


def one_bracket(col, nz):
    """k_colstats_one: float bracket [lof, hif] = edges of the 22-bit float-key bins of the wanted sample ranks"""
    v = col[sample_rows(col.size)]
    v = v[~np.isnan(v)]
    if nz:
        v = v[v != 0]
    with np.errstate(over="ignore"):
        k = np.sort(fkey(v.astype(np.float32)))
    a, b = bracket_ranks(k.size)
    lof, hif = np.float32(-np.inf), np.float32(np.inf)
    if a is not None:
        f = fval(int(k[a]) >> 10 << 10)
        lof = f if f == f else lof
    if b is not None:
        f = fval(int(k[b]) | 1023)
        hif = f if f == f else hif
    return lof, hif


def fast_bracket(col, g):
    """k_colstats_fast: bracket [lo, hi] = sample values of the wanted ranks (g = 0 all values, 1 non-zero)"""
    v = col[sample_rows(col.size)]
    k = np.sort(dkey(v[~np.isnan(v)]))
    zero = np.uint64(1 << 63)
    zs, ze = int(np.searchsorted(k, zero, "left")), int(np.searchsorted(k, zero, "right"))
    m = k.size - (ze - zs if g else 0)
    a, b = bracket_ranks(m)
    lo, hi = -np.inf, np.inf
    if a is not None:
        lo = kval(k[a + (ze - zs if g and a >= zs else 0)])
    if b is not None:
        hi = kval(k[b + (ze - zs if g and b >= zs else 0)])
    return lo, hi


def kval(k):
    k = np.uint64(k)
    b = k & np.uint64(0x7FFFFFFFFFFFFFFF) if k >> np.uint64(63) else ~k
    return float(np.array(b, dtype=np.uint64).view(np.float64))


def thread_rows(S):
    """rows[t, i] = i-th row thread t of a column CTA reads (-1 past the end)"""
    r = np.arange(NT)[:, None] + NT * np.arange((S + NT - 1) // NT)[None, :]
    return np.where(r < S, r, -1)


def route_model(col, kernel):
    """True when the one-pass kernel `kernel` ("one_all", "one_nz" or "two") accepts the column (no redo)"""
    S = col.size
    nan = np.isnan(col)
    with np.errstate(over="ignore", invalid="ignore"):
        if kernel == "two":
            for g in (0, 1):
                lo, hi = fast_bracket(col, g)
                live = ~nan & ((col != 0) if g else True)
                inside = live & (col > lo) & (col < hi)
                warp = (np.arange(S) % NT) // 32
                if np.bincount(warp[inside], minlength=8).max() > WCAP:
                    return False
                n = int(live.sum())
                if n == 0:
                    continue
                below, eqlo = int((live & (col < lo)).sum()), int((live & (col == lo)).sum())
                eqhi = int((live & (col == hi)).sum()) if hi != lo else 0
                ka, kb = ranks(n)
                if ka < below or kb >= below + eqlo + int(inside.sum()) + eqhi:
                    return False
            return True
        nz = kernel == "one_nz"
        if nan.any():
            return False  # a NaN row is always a candidate
        lof, hif = one_bracket(col, nz)
        f = col.astype(np.float32)
        isz = col == 0
        cd = ~((f < lof) | (f > hif))
        if nz and lof <= 0 <= hif:
            cd &= ~isz
        below = int((f < lof).sum()) - (int(isz.sum()) if nz and lof > 0 else 0)
        count = S - (int(isz.sum()) if nz else 0)
        # private slots: flushed to the shared overflow area when more than 16 are taken before a group of 4 rows
        # (8 rows per thread and 2048-row block), then, in the tail past the last full block, when all 20 are taken
        tr = thread_rows(S)
        c = np.where(tr >= 0, cd[np.maximum(tr, 0)], False).astype(np.int64)
        cnt, novf = np.zeros(NT, np.int64), 0
        main = (S // (NT * 8)) * 8
        for i0 in range(0, main, 4):
            fl = cnt > TCAP - 4
            novf += int(cnt[fl].sum())
            cnt[fl] = 0
            cnt += c[:, i0:i0 + 4].sum(1)
        for i in range(main, c.shape[1]):
            fl = (cnt >= TCAP) & (tr[:, i] >= 0)
            novf += int(cnt[fl].sum())
            cnt[fl] = 0
            cnt += c[:, i]
        if novf > OVF:
            return False
        if count == 0:
            return True
        ka, kb = ranks(count)
        return below <= ka and kb < below + int(cd.sum())


# ---- the catalogue ---------------------------------------------------------------------------------------------
def _spread(rng, vals, S, rows=None):
    """a column holding vals on `rows` (default: all rows) in random order"""
    col = np.empty(S)
    rows = np.arange(S) if rows is None else rows
    col[rows] = rng.permutation(vals)
    return col


def _distinct_normal(rng, n):
    v = np.unique(rng.normal(size=n + 64))
    v = v[v != 0]
    return rng.permutation(v)[:n]


def _quantile_sampled(v, rng):
    """the sorted values v as a column whose sampled rows hold exactly the values of their own rank (the sample is
    the column's quantiles, so where the bracket falls is known); every other row in random order"""
    S = v.size
    col = np.sort(v)
    other = np.setdiff1d(np.arange(S), sample_rows(S))
    col[other] = rng.permutation(col[other])
    return col


def _sorted_middles(col):
    v = np.sort(col[~np.isnan(col)])
    ka, kb = ranks(v.size)
    return v, ka, kb


def k_normal(S, rng):
    # ordinary: every one-pass kernel accepts, candidates well under every cap
    return rng.normal(size=S)


def k_abs_zeros30(S, rng):
    # ordinary with zeros: the non-zero bracket lies above the zeros (lof > 0, the zeros counted below, then removed)
    col = np.abs(rng.normal(size=S))
    col[rng.random(S) < 0.3] = 0.0
    assert np.mean(col == 0) > 0.2
    return col


def k_all_negative(S, rng):
    # ordinary, negative keys only (the sign flip of key_of / fkey)
    return -np.abs(rng.normal(size=S)) - 1.0


def k_narrow(S, rng):
    # 3 + k ulp(3): neighbouring order statistics are 1 ulp apart, and all of them round to one float
    ulp = np.spacing(3.0)
    col = 3.0 + rng.integers(0, 200, size=S) * ulp
    assert np.array_equal(np.diff(np.unique(col)), np.full(np.unique(col).size - 1, ulp))
    return col


def k_even_b_is_a(S, rng):
    # even count: the lower middle has one copy at the upper middle, so B = A (qb < cle in the successor scan)
    v = np.sort(_distinct_normal(rng, S))
    ka, kb = ranks(S)
    v[kb] = v[ka]
    if S % 2 == 0:
        assert v[ka] == v[kb] and v[ka - 1] < v[ka] < v[kb + 1]
    return _quantile_sampled(v, rng)


def k_even_b_is_next(S, rng):
    # even count: five copies of the lower middle end at rank ka, so B is the next key (nxt of the successor scan)
    v = np.sort(_distinct_normal(rng, S))
    ka, kb = ranks(S)
    v[ka - 4:ka + 1] = v[ka]
    if S % 2 == 0:
        assert v[ka - 4] == v[ka] < v[kb] and v[ka - 5] < v[ka]
    return _quantile_sampled(v, rng)


def k_copies_100(S, rng):
    # 100 copies of the median key: more than 64, so the radix select of k_colstats_one decides every bit (hi_bit < 0)
    v = np.sort(_distinct_normal(rng, S))
    ka, _ = ranks(S)
    v[ka - 50:ka + 50] = v[ka]
    w, a, b = _sorted_middles(v)
    assert w[a] == w[b] and np.sum(w == w[a]) == 100
    return _quantile_sampled(v, rng)


def k_copies_400(S, rng):
    # 400 copies of the median key: more than CAND = 256, so k_colstats refines down to the last digit
    v = np.sort(_distinct_normal(rng, S))
    ka, _ = ranks(S)
    v[ka - 200:ka + 200] = v[ka]
    assert np.sum(v == v[ka]) == 400
    return _quantile_sampled(v, rng)


def k_eqlo(S, rng):
    # k_colstats_fast: the lower middle equals the bracket's lo sample value (copies end at rank ka, counted in
    # eqlo) while the upper middle lies strictly inside the bracket
    v = np.sort(_distinct_normal(rng, S))
    ka, kb = ranks(S)
    v[ka - S // 8:ka + 1] = v[ka]
    col = _quantile_sampled(v, rng)
    lo, hi = fast_bracket(col, 0)
    assert lo == v[ka] and (S % 2 == 1 or lo < v[kb] < hi), (lo, hi)
    return col


def k_eqhi(S, rng):
    # k_colstats_fast: the upper middle equals the bracket's hi sample value (copies start at rank kb, eqhi) while
    # the lower middle lies strictly inside the bracket
    v = np.sort(_distinct_normal(rng, S))
    ka, kb = ranks(S)
    v[kb:kb + S // 8] = v[kb]
    col = _quantile_sampled(v, rng)
    lo, hi = fast_bracket(col, 0)
    assert hi == v[kb] and (S % 2 == 1 or lo < v[ka] < hi), (lo, hi)
    return col


def k_collapsed(S, rng):
    # every sampled row holds the lower middle: lo == hi, and (even S) the upper middle lies past the copies, so
    # the kernels must reject (k_colstats_fast counts the copies in eqlo only, never again in eqhi)
    v = np.sort(_distinct_normal(rng, S))
    ka, kb = ranks(S)
    v[ka - SAMP + 1:ka + 1] = v[ka]
    col = np.empty(S)
    srow = sample_rows(S)
    rest = np.setdiff1d(np.arange(S), srow)
    col[srow] = v[ka]
    col[rest] = rng.permutation(np.concatenate([v[:ka - SAMP + 1], v[ka + 1:]]))
    lo, hi = fast_bracket(col, 0)
    assert lo == hi == v[ka] and (S % 2 == 1 or v[kb] > v[ka])
    return col


def k_collapsed_zero(S, rng):
    # S = 4096: the sampled rows (every 4th) hold the zeros, which end at rank ka; the rest are distinct non-zeros
    # whose own bracket is the whole line (no non-zero sample point).  The all-values bracket is lo == hi == 0 with
    # the upper middle past it, and since the non-zero median is accepted, only that bracket decides the reject
    assert S == 4096
    ka, kb = ranks(S)
    col = np.zeros(S)
    rest = np.setdiff1d(np.arange(S), sample_rows(S))
    col[rest] = rng.permutation(np.concatenate([-1.0 - rng.random(ka + 1 - SAMP), 1.0 + rng.random(S - ka - 1)]))
    w = np.sort(col)
    assert fast_bracket(col, 0) == (0.0, 0.0) and w[ka] == 0 and w[kb] >= 1
    return col


def k_bracket_miss(S, rng):
    # the sampled rows carry values far above the rest: the true median lies below the bracket
    col = rng.normal(size=S)
    col[sample_rows(S)] = 100.0 + rng.random(SAMP)
    w, ka, _ = _sorted_middles(col)
    assert w[ka] < fast_bracket(col, 0)[0] and w[ka] < one_bracket(col, False)[0]
    return col


def k_float_end_doubles(S, rng):
    # distinct doubles that round to the float of a bracket end: 100 around each end of both brackets, on rows the
    # sample does not read (the fp32 filter cannot decide them, the exact tests must)
    col = rng.normal(size=S)
    free = rng.permutation(np.setdiff1d(np.arange(S), sample_rows(S)))
    lof, hif = one_bracket(col, False)
    lo, hi = fast_bracket(col, 0)
    near = []
    for e in (float(lof), float(hif), lo, hi):
        near.append(e + np.arange(-50, 50) * np.spacing(e))
    near = np.concatenate(near)
    col[free[:near.size]] = near
    assert one_bracket(col, False) == (lof, hif) and fast_bracket(col, 0) == (lo, hi)
    assert np.sum(near.astype(np.float32) == lof) >= 100 and np.sum(near.astype(np.float32) == hif) >= 100
    return col


def k_beyond_float(S, rng):
    # every value beyond the float range: rn(v) = +-inf for every row
    col = rng.normal(size=S) * 1e200
    with np.errstate(over="ignore"):
        assert np.all(np.isinf(col.astype(np.float32)))
    return col


def k_float_subnormal(S, rng):
    # positive values in the float-subnormal range (float keys 2^-149 apart)
    col = (rng.random(S) + 0.01) * 2.0 ** -140
    assert col.min() > 0 and col.astype(np.float32).max() < np.finfo(np.float32).tiny
    return col


def k_infinities(S, rng):
    # +-inf on 10 % of the rows each, finite median
    col = rng.normal(size=S)
    u = rng.random(S)
    col[u < 0.1] = np.inf
    col[u > 0.9] = -np.inf
    w, ka, kb = _sorted_middles(col)
    assert np.isfinite(w[ka]) and np.isfinite(w[kb])
    return col


def k_inf_middles(S, rng):
    # half -inf, half +inf: the middles are -inf and +inf and the median is NaN (odd S: one zero in the middle)
    h = S // 2
    col = _spread(rng, np.concatenate([np.full(h, -np.inf), np.full(h, np.inf), np.zeros(S - 2 * h)]), S)
    w, ka, kb = _sorted_middles(col)
    assert S % 2 == 1 or (w[ka] == -np.inf and w[kb] == np.inf)
    return col


def k_signed_zeros(S, rng):
    # signed zeros only: the median is 0 (key_of maps -0 to +0), the non-zero median of nothing is 0
    col = np.where(rng.random(S) < 0.5, 0.0, -0.0)
    assert np.signbit(col).any() and not np.signbit(col).all()
    return col


def k_zeros_below(S, rng):
    # 60 % zeros, non-zeros in [1, 2]: the non-zero bracket lies above the zeros (lof > 0)
    col = 1.0 + rng.random(S)
    col[rng.random(S) < 0.6] = 0.0
    assert one_bracket(col, True)[0] > 0
    return col


def k_zeros_inside(S, rng):
    # normal with 30 % zeros: the zeros lie inside the non-zero bracket (zin: counted, never candidates)
    col = rng.normal(size=S)
    col[rng.random(S) < 0.3] = 0.0
    col = _quantile_sampled(col, rng)
    lof, hif = one_bracket(col, True)
    assert lof <= 0 <= hif
    return col


def k_zeros_above(S, rng):
    # negative non-zeros with 30 % zeros: the non-zero bracket lies below the zeros (hif < 0)
    col = -np.abs(rng.normal(size=S)) - 0.1
    col[rng.random(S) < 0.3] = 0.0
    assert one_bracket(col, True)[1] < 0
    return col


def k_tiny_nonzeros(S, rng):
    # 40 % zeros and 10 % +-1e-50: non-zero values whose float is +-0 (the zero test must look at the double)
    col = np.abs(rng.normal(size=S))
    u = rng.random(S)
    col[u < 0.4] = 0.0
    col[(u >= 0.4) & (u < 0.45)] = 1e-50
    col[(u >= 0.45) & (u < 0.5)] = -1e-50
    assert np.all(np.float32(col[np.abs(col) == 1e-50]) == 0)
    return col


def k_few_nonzeros(S, rng):
    # 30 non-zeros among zeros: fewer than 48 non-zero sample points (the bracket is the whole line)
    col = np.zeros(S)
    col[rng.choice(S, 30, replace=False)] = rng.random(30) + 0.5
    assert np.count_nonzero(col[sample_rows(S)]) < 48
    return col


def k_all_zero(S, rng):
    # all zero: the median over the non-zeros is 0 by definition
    return np.zeros(S)


def k_one_nan(S, rng):
    # one NaN on a row the sample does not read: the one-median kernel rejects the column, the two-median one drops it
    col = rng.normal(size=S)
    r = int(rng.choice(np.setdiff1d(np.arange(S), sample_rows(S))))
    col[r] = np.nan
    return col


def k_all_nan(S, rng):
    # all NaN: median NaN, non-zero median 0, column minimum +inf
    return np.full(S, np.nan)


def k_nan_sampled(S, rng):
    # NaN on exactly the sampled rows: the sample holds no valid value
    col = rng.normal(size=S)
    col[sample_rows(S)] = np.nan
    assert np.isnan(col).sum() == SAMP
    return col


def _near_zero_column(S, rng, inner, outer):
    """the capacity design: the rows of mask `inner` (never sampled) hold distinct values in (-1e-3, 1e-3), rising
    with the row; every other row holds outer(n, sign, sampled), as many negative as positive values, and the
    sampled rows alternate in sign, so the brackets of both one-pass kernels span the near-zero values and the
    median falls among them"""
    srow = sample_rows(S)
    assert S == S_CAP and not inner[srow].any()
    n_in = int(inner.sum())
    n_neg = (S - n_in) // 2
    col = np.empty(S)
    col[srow[0::2]], col[srow[1::2]] = outer(SAMP // 2, -1.0, True), outer(SAMP // 2, 1.0, True)
    rest = ~inner
    rest[srow] = False
    col[rest] = rng.permutation(np.concatenate([outer(n_neg - SAMP // 2, -1.0, False),
                                                outer(S - n_in - n_neg - SAMP // 2, 1.0, False)]))
    col[inner] = np.sort(rng.uniform(-1e-3, 1e-3, size=n_in))
    assert np.unique(col[inner]).size == n_in and np.all(col[inner] != 0)
    w, ka, kb = _sorted_middles(col)
    assert np.abs(w[ka]) < 1e-3 and np.abs(w[kb]) < 1e-3
    return col


def _residues(S, res):
    return np.isin(np.arange(S) % NT, res)


def _distinct(rng):
    """distinct values: the sampled ones within 1e-3 of +-1, the others beyond 1.01 in magnitude, so the only rows
    of the bracket besides the near-zero ones are the ~86 sampled rows next to +-1"""
    return lambda n, sign, sampled: sign * (1.0 + rng.random(n) * 1e-3 if sampled else 1.01 + rng.random(n))


def k_overflow_accepted(S, rng):
    # k_colstats_one: thread 5 reads exactly the rows = 5 (mod 256); those 128 rows all lie in the bracket (the median
    # pair among them), so thread 5 flushes 120 of them to the shared overflow area, which stays under OVF: the
    # selection and the successor scan must read the overflow slots
    return _near_zero_column(S, rng, _residues(S, [5]), _distinct(rng))


def k_overflow_rejected(S, rng):
    # the same design on 8 residue classes (5 + 32 w, one per warp): 960 overflow entries, more than OVF
    return _near_zero_column(S, rng, _residues(S, [5 + 32 * w for w in range(8)]), _distinct(rng))


def _warp3(S, k):
    """the first k rows (in row order) among those = 97 .. 127 (mod 256): rows of warp 3, never sampled at S_CAP"""
    rows = np.flatnonzero(_residues(S, np.arange(97, 128)))[:k]
    m = np.zeros(S, bool)
    m[rows] = True
    return m


def _ties(n, sign, sampled):
    return np.full(n, 1.5 * sign)


def k_warp_416(S, rng):
    # k_colstats_fast: every other row is -1.5 or +1.5 (== lo or == hi, never in the bracket), and exactly WCAP rows
    # of warp 3 lie strictly inside the bracket: the warp's candidate segment is full, not overflowing
    return _near_zero_column(S, rng, _warp3(S, WCAP), _ties)


def k_warp_417(S, rng):
    # one row more than WCAP inside the bracket on warp 3's rows: the two-median kernel rejects the column
    return _near_zero_column(S, rng, _warp3(S, WCAP + 1), _ties)


# name -> generator; the capacity kinds are designed for S_CAP rows only
CATALOGUE = {f.__name__[2:]: f for f in [
    k_normal, k_abs_zeros30, k_all_negative, k_narrow, k_even_b_is_a, k_even_b_is_next, k_copies_100, k_copies_400,
    k_eqlo, k_eqhi, k_collapsed, k_collapsed_zero, k_bracket_miss, k_float_end_doubles, k_beyond_float, k_float_subnormal,
    k_infinities, k_inf_middles, k_signed_zeros, k_zeros_below, k_zeros_inside, k_zeros_above, k_tiny_nonzeros,
    k_few_nonzeros, k_all_zero, k_one_nan, k_all_nan, k_nan_sampled,
    k_overflow_accepted, k_overflow_rejected, k_warp_416, k_warp_417]}
# kinds designed for one column length only
SPECIAL = {"overflow_accepted": S_CAP, "overflow_rejected": S_CAP, "warp_416": S_CAP, "warp_417": S_CAP,
           "collapsed_zero": 4096}
GENERAL = [k for k in CATALOGUE if k not in SPECIAL]

# Which one-pass kernel accepts (A: computes the medians itself) or rejects (R: hands the column to k_colstats)
# each kind: (k_colstats_one<false>, k_colstats_one<true>, k_colstats_fast<true, true>).  A rewrite of the
# statistics pass that changes what it accepts updates this table on purpose; the values are checked bit for bit
# whatever the route.
ROUTES = {
    "normal": "AAA", "abs_zeros30": "AAA", "all_negative": "AAA",
    "narrow": "RRA",             # one float for every value: all rows are float-bracket candidates
    "even_b_is_a": "AAA", "even_b_is_next": "AAA", "copies_100": "AAA", "copies_400": "AAA",
    "eqlo": "RRA", "eqhi": "RRA",  # S/8 copies of one key overflow the one-median candidate slots
    "collapsed": "RRR", "collapsed_zero": "RAR", "bracket_miss": "RRR",
    "float_end_doubles": "AAA",
    "beyond_float": "RRA", "float_subnormal": "RRA",  # every row in one or two float bins
    "infinities": "AAA",
    "inf_middles": "RRA",
    "signed_zeros": "RAA", "zeros_below": "RAA", "zeros_inside": "RAA", "zeros_above": "AAA",
    "tiny_nonzeros": "RAA", "few_nonzeros": "RAA", "all_zero": "RAA",
    "one_nan": "RRA", "all_nan": "RRA", "nan_sampled": "RRR",
    "overflow_accepted": "AAA", "overflow_rejected": "RRA",
    "warp_416": "RRA", "warp_417": "RRR",
}
KERNELS = ("one_all", "one_nz", "two")


def kinds_at(S):
    return [k for k, s in SPECIAL.items() if s == S] + (GENERAL if S in SHAPES else [])


def column(kind, S, seed=0):
    return CATALOGUE[kind](S, np.random.default_rng([seed, S, sorted(CATALOGUE).index(kind)]))


# ---- reference -------------------------------------------------------------------------------------------------
def ref_stats(x):
    """med_all (NaN dropped), med_nz (NaN and zeros dropped, empty -> 0), colmin (+inf when all NaN)"""
    med_all = O.col_medians_narm(x)
    z = np.where(x == 0, np.nan, x)
    med_nz = O.col_medians_narm(z)
    med_nz[np.isnan(med_nz)] = 0.0
    with np.errstate(invalid="ignore"):
        colmin = np.array([np.min(c[~np.isnan(c)]) if (~np.isnan(c)).any() else np.inf for c in x.T])
    return med_all, med_nz, colmin


def model_normalized(x, iz=None):
    """normalize_medians: x + (c - med) in that order (the __dadd_rn sequence of k_fixup, alpha = 1)"""
    med_all, med_nz, colmin = ref_stats(x)
    if iz is None:
        iz = bool(np.min(colmin) == 0)
    med = med_nz if iz else med_all
    c = O.r_mean(med)
    with np.errstate(invalid="ignore"):
        return x + (c - med)[None, :]


def same_bits(got, want, what):
    """bit for bit, NaN by isnan, -0 == +0; names the first differing entry"""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, what
    g = np.where(got == 0, 0.0, got)
    w = np.where(want == 0, 0.0, want)
    bad = (g.view(np.int64) != w.view(np.int64)) & ~(np.isnan(g) & np.isnan(w))
    if bad.any():
        i = np.unravel_index(np.flatnonzero(bad)[0], bad.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} entries differ, first at {i}: got {g[i]!r}, want {w[i]!r}")


def matrix(kinds, S, seed=0):
    return np.asfortranarray(np.column_stack([column(k, S, seed) for k in kinds]))


def groups(kinds, n):
    return [kinds[i:i + n] for i in range(0, len(kinds), n)]


# ---- CPU rehearsal of the catalogue ----------------------------------------------------------------------------
def test_catalogue_self_checks():
    """every generator's own checks at every shape, and the route table against route_model (no GPU needed)"""
    for S in SHAPES:
        for kind in GENERAL:
            col = column(kind, S)
            assert col.shape == (S,), kind
    for kind in CATALOGUE:
        S = SPECIAL.get(kind, S_ROUTE)
        for seed in range(4):
            col = column(kind, S, seed)
            got = "".join("A" if route_model(col, k) else "R" for k in KERNELS)
            assert got == ROUTES[kind], (kind, seed, got)


# ---- GPU: normalize_medians bit for bit -------------------------------------------------------------------------
def normalize(ctx, x, iz):
    from plaid_b200 import _lib as L
    res = np.empty_like(x, order="F")
    ctx.check(ctx.lib.plaidgpu_normalize_medians(ctx.h, x.ctypes.data, x.shape[0], x.shape[1], iz, L.HOST,
                                                 res.ctypes.data))
    return res


@pytest.mark.parametrize("S", SHAPES + (S_CAP,))
def test_normalize_medians_bit_exact(gpu_ctx, S):
    """plaidgpu_normalize_medians (ignore.zero NULL / FALSE / TRUE) against x + (c - med); N = 1, 2 and 7 columns
    per launch: k_fixup_flat chunks that straddle column boundaries (6144 < S), one column per chunk (S = 4096), a
    partial last chunk; k_fixup with odd S on both 16-byte alignments of a column"""
    kinds = kinds_at(S)
    for n in (1, 2, 7):
        for ks in groups(kinds, n):
            x = matrix(ks, S, seed=n)
            for iz in (-1, 0, 1):
                same_bits(normalize(gpu_ctx, x, iz), model_normalized(x, None if iz < 0 else bool(iz)),
                          f"S={S} iz={iz} columns={ks}")


def test_normalize_medians_many_columns_per_cta(gpu_ctx):
    """S = 4096 and 1,600 columns: more columns than CTAs (148 SMs x at most 8), so each CTA walks several; the
    kinds are interleaved, so a rejected or overflowing column is followed by ordinary ones in the same CTA"""
    S = 4096
    kinds = [GENERAL[j % len(GENERAL)] for j in range(1600)]
    x = np.asfortranarray(np.column_stack([column(k, S, seed=j) for j, k in enumerate(kinds)]))
    for iz in (-1, 0, 1):
        same_bits(normalize(gpu_ctx, x, iz), model_normalized(x, None if iz < 0 else bool(iz)), f"iz={iz}")
    score_medians(x, "many columns")


# ---- GPU: the medians of a scoring call --------------------------------------------------------------------------
def score_medians(x, label, tiled_budget=None, monkeypatch=None):
    """x scored with one gene set per gene (G = I, stats = "sum", fp64 adds): the raw scores are x itself.  Checks
    that, then both median vectors and score_min of plaidgpu_score_begin / _compute / get_col_medians, and the
    normalised output of _finish, bit for bit"""
    import plaid_b200 as pb
    from plaid_b200 import _lib as L
    from plaid_b200.api import _matrix_struct, _opts
    S, N = x.shape
    ctx = pb.Context(0)
    try:
        ctx.set_genesets(sp.identity(S, format="csc"))
        rowmap = np.arange(S, dtype=np.int32)
        keep = []
        M = _matrix_struct(x, keep)
        raw = np.empty((S, N), order="F")
        o = _opts(ctx.lib, scorer=L.PLAID, stats_mean=0, normalize=0, exact_fp64=1, out_location=L.HOST)
        ctx.check(ctx.lib.plaidgpu_score(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), raw.ctypes.data))
        same_bits(raw, x, f"{label}: raw scores of G = I")
        med_all, med_nz, colmin = ref_stats(x)
        want = model_normalized(x)
        o = _opts(ctx.lib, scorer=L.PLAID, stats_mean=0, normalize=1, ignore_zero=-1, exact_fp64=1, out_location=L.HOST)
        out = np.empty((S, N), order="F")
        if tiled_budget is not None:  # column tiles, both medians per tile (k_colstats_fast<true, true>)
            monkeypatch.setenv("PLAIDGPU_MAX_OUT_BYTES", str(tiled_budget))
            try:
                ctx.check(ctx.lib.plaidgpu_score(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), out.ctypes.data))
            finally:
                monkeypatch.delenv("PLAIDGPU_MAX_OUT_BYTES")
            same_bits(out, want, f"{label}: normalised output of the column-tiled call")
            return
        loc = L.Scalars()
        ctx.check(ctx.lib.plaidgpu_score_begin(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), C.byref(loc)))
        ctx.check(ctx.lib.plaidgpu_score_compute(ctx.h, C.byref(loc), None))
        ma, mz = np.empty(N), np.empty(N)
        ctx.check(ctx.lib.plaidgpu_get_col_medians(ctx.h, ma.ctypes.data, mz.ctypes.data))
        same_bits(ma, med_all, f"{label}: med_all")
        same_bits(mz, med_nz, f"{label}: med_nz")
        same_bits(loc.score_min, np.min(colmin), f"{label}: score_min")
        scal = L.Scalars()
        ctx.check(ctx.lib.plaidgpu_combine_medians(-1, loc.score_min, ma.ctypes.data, mz.ctypes.data, N, C.byref(scal)))
        ctx.check(ctx.lib.plaidgpu_score_finish(ctx.h, C.byref(scal), out.ctypes.data))
        same_bits(out, want, f"{label}: normalised output")
    finally:
        ctx.close()


def min_sign(col):
    with np.errstate(invalid="ignore"):
        m = np.nanmin(col) if (~np.isnan(col)).any() else np.inf
    return int(np.sign(m))


@pytest.mark.parametrize("S", SHAPES + (S_CAP,))
def test_scoring_medians_bit_exact(S):
    """both median vectors of a scoring call: the shard's minimum picks the kernel (> 0: the plain median, copied
    into the non-zero one; == 0: the non-zero median; < 0: the plain median) and the other one is computed on
    demand; one call per sign of the minimum"""
    kinds = kinds_at(S)
    cols = {k: column(k, S, seed=3) for k in kinds}
    for sign in (1, 0, -1):
        ks = [k for k in kinds if min_sign(cols[k]) == sign]
        if sign == 1:  # an ordinary column without zeros next to the few positive kinds
            cols["abs_normal_plus"] = np.abs(np.random.default_rng([S, 9]).normal(size=S)) + 0.5
            ks.append("abs_normal_plus")
        if ks:
            score_medians(np.asfortranarray(np.column_stack([cols[k] for k in ks])), f"S={S} min sign {sign} {ks}")


def test_scoring_column_tiled_bit_exact(monkeypatch):
    """a normalised call larger than its output budget: tiles of 3 columns, both medians of every tile in one
    launch of the two-median kernel; the normalised output equals the model bit for bit"""
    S = S_ROUTE
    x = matrix(GENERAL, S, seed=4)
    score_medians(x, "tiled", tiled_budget=S * 8 * 3, monkeypatch=monkeypatch)


# ---- GPU: which kernel took which column -------------------------------------------------------------------------
REDONE = re.compile(r"colstats: (\d+) of (\d+) columns redone")


def redone(ctx, x, iz, monkeypatch, capfd):
    monkeypatch.setenv("PLAIDGPU_TRACE_COLSTATS", "1")
    try:
        capfd.readouterr()
        got = normalize(ctx, x, iz)
        err = capfd.readouterr().err
    finally:
        monkeypatch.delenv("PLAIDGPU_TRACE_COLSTATS")
    same_bits(got, model_normalized(x, None if iz < 0 else bool(iz)), f"iz={iz}")
    m = REDONE.findall(err)
    assert len(m) == 1 and int(m[0][1]) == x.shape[1], err
    return int(m[0][0])


def test_route_table(gpu_ctx, monkeypatch, capfd):
    """one launch of 4 columns (4 seeds) per kind and one-pass kernel: an accepting kernel redoes none of them,
    a rejecting one all four"""
    iz_of = {"one_all": 0, "one_nz": 1, "two": -1}
    failures = []
    for kind in CATALOGUE:
        S = SPECIAL.get(kind, S_ROUTE)
        x = np.asfortranarray(np.column_stack([column(kind, S, seed) for seed in range(4)]))
        for kernel, want in zip(KERNELS, ROUTES[kind]):
            n = redone(gpu_ctx, x, iz_of[kernel], monkeypatch, capfd)
            if n != (0 if want == "A" else 4):
                failures.append(f"{kind} {kernel}: {n} of 4 redone, table says {want}")
    assert not failures, failures


def test_redone_share_at_70000_rows(gpu_ctx, monkeypatch, capfd):
    """not asserted: how many ordinary columns of 70,000 rows each one-pass kernel hands to the three-pass kernel"""
    x = np.asfortranarray(np.random.default_rng(70000).normal(size=(70000, 256)))
    counts = {kernel: redone(gpu_ctx, x, iz, monkeypatch, capfd) for kernel, iz in (("one_all", 0), ("two", -1))}
    with capfd.disabled():
        print(f"\nS=70000, 256 normal columns, redone by the three-pass kernel: {counts}")
