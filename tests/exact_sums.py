"""Exact co-rating sums of integer ratings, and the similarities the tensor path forms from them, on the CPU.

The six sums of every pair (a, b) of left rows are integer products of the rating planes X (the rating), X2 (its
square) and M (1 where rated), as the tensor path forms them on the device (csrc/sim_tensor.cu):
    count = M M^T   Sx = X M^T   Sy = M X^T = Sx^T   Sxx = X2 M^T   Syy = Sxx^T   Sxy = X X^T
computed here with scipy.sparse in int64, independently of the oracle.  From them:
  - Pearson as pearson_from_sums defines it, L / (sqrt(Mi) sqrt(Ni)) with
        Mi = ca^2 Sxx - 2 ca sa Sx + n sa^2,  Ni = cb^2 Syy - 2 cb sb Sy + n sb^2,
        L  = ca cb Sxy - ca sb Sx - cb sa Sy + n sa sb          (ca, sa: count and sum of row a)
    as an exact integer triple and its value to 64 bits of mantissa: np.longdouble while |L|, Mi and Ni are below
    2^63, decimal at 50 digits beyond (Python ints hold the triple at any size);
  - Cosine and MSD with the reference's float64 operations (core/sim.go), in numpy: below 2^53 the sums are exact
    doubles, so this is the oracle's value bit for bit at any K, where the oracle itself is too slow;
  - ulp distances of a float64 result from an exact value, and the rules a tensor-path Pearson must meet."""
import decimal

import numpy as np
import scipy.sparse as sp

TWO53 = 1 << 53
TWO63 = 1 << 63
# Derived bounds, not measured ones.  |L|, Mi and Ni < 2^53: they convert exactly, and two square roots, a product and a
# quotient each round once to nearest: relative error (1 + u)^4 - 1 = 4u + O(u^2), u = 2^-53, and the float64 ulp at
# x exceeds u |x|.  Beyond: the conversions round to nearest too (pearson_from_sums converts __int128 explicitly), that
# of L adds u, those of Mi and Ni u each, halved by the square root.  The second-order terms are below 2^-48 ulps.
MAX_ULPS_SMALL = 4 + 2.0 ** -48
MAX_ULPS_LARGE = 6 + 2.0 ** -48

assert np.finfo(np.longdouble).nmant >= 63, "the exact reference needs an 80-bit long double (x86-64)"


class Sums:
    """The exact sums of every pair of left rows (n_left x n_left int64 arrays) and each row's count and sum."""

    def __init__(self, left, right, rating, n_left, n_right):
        r = np.asarray(rating, dtype=np.float64)
        x = r.astype(np.int64)
        assert np.array_equal(x, r) and np.abs(x).max() <= 11, "integer ratings in [-11, 11] only"
        left, right = np.asarray(left, dtype=np.int64), np.asarray(right, dtype=np.int64)

        def plane(v):
            return sp.csr_matrix((v, (left, right)), shape=(n_left, n_right), dtype=np.int64)

        M, X, X2 = plane(np.ones_like(x)), plane(x), plane(x * x)
        self.n = (M @ M.T).toarray()
        self.sx = (X @ M.T).toarray()
        self.sy = self.sx.T.copy()
        self.sxx = (X2 @ M.T).toarray()
        self.syy = self.sxx.T.copy()
        self.sxy = (X @ X.T).toarray()
        self.row_cnt = np.asarray(M.sum(axis=1)).ravel()
        self.row_sum = np.asarray(X.sum(axis=1)).ravel()
        self.max_abs = int(np.abs(x).max())

    def six(self, a, b):
        """(count, Sx, Sy, Sxx, Syy, Sxy) of the pair, the layout of the oracle's pair_sums and rs_knn_cosums."""
        return np.array([s[a, b] for s in (self.n, self.sx, self.sy, self.sxx, self.syy, self.sxy)], dtype=np.int64)

    # ---- Pearson `sums` ----
    def pearson_terms(self):
        """(L, Mi, Ni) of every pair: int64 arrays when every partial term provably fits int64 (each is at most
        c^3 m^2 for rows of at most c ratings of |x| <= m, four of them), else object arrays of Python ints."""
        c, m = int(self.row_cnt.max()), self.max_abs
        fits = 4 * c ** 3 * m * m < TWO63
        conv = (lambda a: a) if fits else (lambda a: a.astype(object))
        n, sx, sy, sxx, syy, sxy = (conv(s) for s in (self.n, self.sx, self.sy, self.sxx, self.syy, self.sxy))
        ca, sa = conv(self.row_cnt)[:, None], conv(self.row_sum)[:, None]
        cb, sb = ca.T, sa.T
        Mi = ca * ca * sxx - 2 * ca * sa * sx + n * sa * sa
        Ni = cb * cb * syy - 2 * cb * sb * sy + n * sb * sb
        L = ca * cb * sxy - ca * sb * sx - cb * sa * sy + n * sa * sb
        return L, Mi, Ni


def pearson_exact(L, Mi, Ni, branch="auto"):
    """L / sqrt(Mi Ni) to 64 bits of mantissa (np.longdouble), NaN where Mi Ni == 0.  branch: "longdouble" (valid
    while |L|, Mi, Ni < 2^63, where the integers convert exactly), "decimal" (50 digits, any size) or "auto" (the
    first where it is valid, else the second)."""
    L, Mi, Ni = (np.asarray(a, dtype=object).ravel() for a in (L, Mi, Ni))
    shape = np.shape(L)
    out = np.full(len(L), np.nan, dtype=np.longdouble)
    ctx = decimal.Context(prec=50)
    for e in range(len(L)):
        l, mi, ni = int(L[e]), int(Mi[e]), int(Ni[e])
        if mi == 0 or ni == 0:
            continue
        small = max(abs(l), mi, ni) < TWO63
        if branch == "longdouble" or (branch == "auto" and small):
            assert small, "the longdouble branch needs |L|, Mi, Ni < 2^63"
            out[e] = np.longdouble(l) / (np.sqrt(np.longdouble(mi)) * np.sqrt(np.longdouble(ni)))
        else:
            q = ctx.divide(decimal.Decimal(l), ctx.sqrt(ctx.multiply(decimal.Decimal(mi), decimal.Decimal(ni))))
            hi = float(q)                                   # q to ~106 bits as hi + lo, then one rounding
            out[e] = np.longdouble(hi) + np.longdouble(float(ctx.subtract(q, decimal.Decimal(hi))))
    return out.reshape(shape)


def pearson_exact_matrix(L, Mi, Ni):
    """pearson_exact of whole matrices, vectorised in longdouble where every entry is below 2^63."""
    if L.dtype != object:
        Ll, Ml, Nl = (a.astype(np.longdouble) for a in (L, Mi, Ni))
        with np.errstate(divide="ignore", invalid="ignore"):
            out = Ll / (np.sqrt(Ml) * np.sqrt(Nl))
        out[(Mi == 0) | (Ni == 0)] = np.nan
        return out
    return pearson_exact(L, Mi, Ni).reshape(L.shape)


def ulps(got, exact):
    """|got - exact| in units of the float64 ulp at exact (2^(e-53) for |exact| in [2^(e-1), 2^e)); exact zeros:
    0 where got is 0 too, else inf.  got: float64, exact: longdouble, same shape, no NaN."""
    got = np.asarray(got, dtype=np.float64).astype(np.longdouble)
    exact = np.asarray(exact, dtype=np.longdouble)
    _, e = np.frexp(exact)
    unit = np.ldexp(np.ones_like(exact), e.astype(np.int64) - 53)
    d = np.abs(got - exact)
    with np.errstate(divide="ignore", invalid="ignore"):
        out = np.where(exact == 0, np.where(got == 0, 0.0, np.inf), d / unit)
    return out.astype(np.float64)


def check_ratio(got, L, Mi, Ni, row0=0, who=""):
    """The rules of a similarity L / (sqrt(Mi) sqrt(Ni)) computed on the device from exact integers (Pearson `sums`,
    Cosine with L = Sxy, Mi = Sxx, Ni = Syy), for the rows row0 .. row0 + len(got) of the full matrices L, Mi, Ni:
    NaN exactly on the diagonal and where Mi Ni == 0; +0.0 with the sign bit clear exactly where L == 0 elsewhere;
    bit-symmetric when got is the whole matrix; within MAX_ULPS_SMALL ulps of the exact value where |L|, Mi, Ni
    < 2^53, MAX_ULPS_LARGE otherwise.  Returns the largest distance in ulps of each regime, (small, large), -1 where
    a regime has no entry."""
    got = np.asarray(got, dtype=np.float64)
    rows = slice(row0, row0 + got.shape[0])
    L, Mi, Ni = L[rows], Mi[rows], Ni[rows]
    exact = pearson_exact_matrix(L, Mi, Ni)
    want_nan = np.asarray((Mi == 0) | (Ni == 0), dtype=bool)
    r = np.arange(got.shape[0])
    want_nan[r, row0 + r] = True
    assert np.array_equal(np.isnan(got), want_nan), (who, "NaN pattern", np.argwhere(np.isnan(got) != want_nan)[:5])
    fin = ~want_nan
    l_zero = np.asarray(L == 0, dtype=bool) & fin
    assert (got[l_zero] == 0).all() and not np.signbit(got[l_zero]).any(), (who, "L == 0 must give +0.0")
    assert (got[fin & ~l_zero] != 0).all(), (who, "a nonzero L gave 0")
    if row0 == 0 and got.shape[0] == got.shape[1]:
        assert np.array_equal(got.view(np.uint64), got.T.view(np.uint64)), (who, "not bit-symmetric")
    big = np.asarray(np.maximum(np.maximum(abs(L), Mi), Ni) >= TWO53, dtype=bool)
    d = np.zeros(got.shape)
    d[fin] = ulps(got[fin], exact[fin])
    worst = []
    for mask, bound in ((fin & ~big, MAX_ULPS_SMALL), (fin & big, MAX_ULPS_LARGE)):
        w = float(d[mask].max()) if mask.any() else -1.0
        assert w <= bound, (who, "ulps", w, bound, np.argwhere(mask & (d > bound))[:5])
        worst.append(w)
    return tuple(worst)


# ---- Cosine and MSD with the reference's float64 operations ----
def cosine(s):
    """core/sim.go:24  l / (sqrt(m) * sqrt(n)) from the exact sums; NaN on the diagonal (core/knn.go:202)."""
    assert max(s.sxx.max(), s.sxy.max(), -s.sxy.min()) < TWO53
    with np.errstate(divide="ignore", invalid="ignore"):
        out = s.sxy.astype(np.float64) / (np.sqrt(s.sxx.astype(np.float64)) * np.sqrt(s.syy.astype(np.float64)))
    np.fill_diagonal(out, np.nan)
    return out


def msd(s):
    """core/sim.go:43  1 / (sum / count + 1), sum = Sxx + Syy - 2 Sxy (exact); NaN on the diagonal."""
    total = s.sxx + s.syy - 2 * s.sxy
    assert total.max() < TWO53
    with np.errstate(divide="ignore", invalid="ignore"):
        out = 1.0 / (total.astype(np.float64) / s.n.astype(np.float64) + 1.0)
    np.fill_diagonal(out, np.nan)
    return out


def msd_exact(s):
    """The exact MSD n / (sum + n) in longdouble (NaN where n == 0 and on the diagonal)."""
    total = (s.sxx + s.syy - 2 * s.sxy).astype(np.longdouble)
    n = s.n.astype(np.longdouble)
    with np.errstate(divide="ignore", invalid="ignore"):
        out = n / (total + n)
    np.fill_diagonal(out, np.nan)
    return out
