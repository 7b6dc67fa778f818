"""The exact reference of tests/exact_sums.py against the oracle and against exact rational arithmetic (no GPU)."""
import decimal
import math
import random
from fractions import Fraction

import numpy as np
import pytest

import exact_sums as ex
from conftest import ROOT, bits_equal


def _small_set(seed, n_users=60, n_items=40, density=0.3, values=np.arange(-11.0, 12.0)):
    rng = np.random.RandomState(seed)
    uu, ii = np.nonzero(rng.uniform(size=(n_users, n_items)) < density)
    return uu, ii, values[rng.randint(0, len(values), len(uu))]


def test_longdouble_is_wide_enough():
    assert np.finfo(np.longdouble).nmant >= 63


def test_sums_equal_the_oracle():
    if not (ROOT / "oracle" / "libknn_oracle.so").exists():
        pytest.skip("the oracle library is not built")
    from oracle import binding as ob

    u, i, r = _small_set(1)
    for user_based in (True, False):
        ref = ob.KNN(sim="cosine", user_based=user_based).fit(ob.TrainSet(u, i, r))
        left, right = _inner(u, i, user_based)
        n_left, n_right = left.max() + 1, right.max() + 1
        s = ex.Sums(left, right, r, n_left, n_right)
        for a in range(0, n_left, 3):
            for b in range(n_left):
                assert np.array_equal(s.six(a, b), ref.pair_sums(a, b)), (user_based, a, b)
        assert bits_equal(ex.cosine(s), ref.sims(copy=False))
        msd_ref = ob.KNN(sim="msd", user_based=user_based).fit(ob.TrainSet(u, i, r))
        assert bits_equal(ex.msd(s), msd_ref.sims(copy=False))


def _inner(u, i, user_based):
    """Left and right inner ids as the oracle's TrainSet assigns them: first-seen order of the dataset."""
    def first_seen(ids):
        _, first = np.unique(ids, return_index=True)
        order = np.argsort(first)
        lut = np.empty(ids.max() + 1, dtype=np.int64)
        lut[np.unique(ids)[order]] = np.arange(len(order))
        return lut[ids]

    iu, ii = first_seen(u), first_seen(i)
    return (iu, ii) if user_based else (ii, iu)


def _fraction_pearson(L, Mi, Ni):
    """L / sqrt(Mi Ni) to 60 digits from exact rationals: sqrt of the exact product by decimal's correctly rounded sqrt."""
    with decimal.localcontext() as c:
        c.prec = 60
        q = Fraction(L) / Fraction(decimal.Decimal(Mi * Ni).sqrt())
        return decimal.Decimal(q.numerator) / decimal.Decimal(q.denominator)


def test_pearson_equals_rational_evaluation():
    """Pearson from the sums, on random small sets of both orientations, against an independent evaluation from the
    ratings themselves: the means as Fractions, Mi = ca^2 sum (x - mean_a)^2 over the co-rated entries."""
    for seed in range(4):
        u, i, r = _small_set(100 + seed, 25, 30, 0.4)
        s = ex.Sums(u, i, r, u.max() + 1, i.max() + 1)
        L, Mi, Ni = s.pearson_terms()
        exact = ex.pearson_exact_matrix(L, Mi, Ni)
        R = np.full((u.max() + 1, i.max() + 1), np.nan)
        R[u, i] = r
        rng = np.random.RandomState(seed)
        for a, b in rng.randint(0, u.max() + 1, size=(60, 2)):
            ra, rb = R[a][~np.isnan(R[a])], R[b][~np.isnan(R[b])]
            ma, mb = Fraction(int(ra.sum()), len(ra)), Fraction(int(rb.sum()), len(rb))
            co = ~np.isnan(R[a]) & ~np.isnan(R[b])
            xa, xb = [Fraction(int(v)) for v in R[a][co]], [Fraction(int(v)) for v in R[b][co]]
            mi = sum((x - ma) ** 2 for x in xa) * len(ra) ** 2
            ni = sum((y - mb) ** 2 for y in xb) * len(rb) ** 2
            l_ = sum((x - ma) * (y - mb) for x, y in zip(xa, xb)) * len(ra) * len(rb)
            assert mi.denominator == ni.denominator == l_.denominator == 1
            assert (int(L[a, b]), int(Mi[a, b]), int(Ni[a, b])) == (int(l_), int(mi), int(ni)), (seed, a, b)
            if mi == 0 or ni == 0:
                assert np.isnan(exact[a, b])
                continue
            want = _fraction_pearson(int(l_), int(mi), int(ni))
            got = decimal.Decimal(repr(float(exact[a, b])))     # float64 of the longdouble value
            assert abs(got - want) <= abs(want) * decimal.Decimal(2) ** -52, (seed, a, b)
            # the longdouble value itself is within a few 64-bit-mantissa ulps
            assert ex.ulps(np.float64(want), np.longdouble(exact[a, b])) <= 0.51


def test_longdouble_and_decimal_branches_agree():
    """Both branches where both apply (|L|, Mi, Ni < 2^63), up to 2^62 in magnitude, to 2^-60 relative."""
    rng = random.Random(7)
    for bits in (10, 40, 53, 60, 62):
        Mi = [rng.randrange(1, 1 << bits) for _ in range(200)]
        Ni = [rng.randrange(1, 1 << bits) for _ in range(200)]
        L = [rng.choice((-1, 1)) * math.isqrt(m * n) // rng.randrange(1, 9) for m, n in zip(Mi, Ni)]
        assert max(max(Mi), max(Ni), max(abs(x) for x in L)) < ex.TWO63
        a = ex.pearson_exact(L, Mi, Ni, "longdouble")
        b = ex.pearson_exact(L, Mi, Ni, "decimal")
        rel = np.abs((a - b) / b)
        assert (rel <= np.ldexp(np.longdouble(1), -60)).all(), (bits, rel.max())
    # beyond 2^63 the longdouble branch is refused and "auto" takes decimal
    with pytest.raises(AssertionError):
        ex.pearson_exact([1], [ex.TWO63], [1], "longdouble")
    q = ex.pearson_exact([3 * ex.TWO63], [4 * ex.TWO63 * ex.TWO63], [9])      # 3 * 2^63 / (2^64 * 3) = 1/2
    assert q[0] == np.longdouble(0.5)


def test_ulps():
    one = np.longdouble(1)
    assert ex.ulps(np.float64(1.0), one) == 0
    assert ex.ulps(np.nextafter(1.0, 2.0), one) == 1
    assert ex.ulps(np.nextafter(1.0, 0.0), one) == 0.5        # the ulp below 1 is half the one above
    assert ex.ulps(np.float64(-0.75), np.longdouble(-0.75) + np.ldexp(one, -55)) == 0.25
    assert ex.ulps(np.float64(0.0), np.longdouble(0)) == 0 and np.isinf(ex.ulps(np.float64(1e-300), np.longdouble(0)))


def test_check_ratio_catches_a_lost_bit():
    """The ulp rule rejects a result 5 ulps off and the sign rule a -0.0; a correctly rounded one passes."""
    u, i, r = _small_set(3, 30, 50, 0.5)
    s = ex.Sums(u, i, r, u.max() + 1, i.max() + 1)
    L, Mi, Ni = s.pearson_terms()
    exact = ex.pearson_exact_matrix(L, Mi, Ni)
    good = exact.astype(np.float64)
    np.fill_diagonal(good, np.nan)
    assert ex.check_ratio(good, L, Mi, Ni)[0] <= 0.5
    bad = good.copy()
    fin = np.argwhere(~np.isnan(bad) & (L != 0))
    a, b = fin[len(fin) // 2]
    bad[a, b] = bad[b, a] = bad[a, b] * (1 + 5 * 2.0 ** -52)
    with pytest.raises(AssertionError):
        ex.check_ratio(bad, L, Mi, Ni)
    zero = np.argwhere(~np.isnan(good) & (L == 0))
    if len(zero):
        bad = good.copy()
        a, b = zero[0]
        bad[a, b] = bad[b, a] = -0.0
        with pytest.raises(AssertionError):
            ex.check_ratio(bad, L, Mi, Ni)
