"""The tensor path at the limits of its integer arithmetic, against the exact reference of tests/exact_sums.py.

Long rows: Pearson `sums` forms Mi, Ni and L (pearson_from_sums, csrc/sim_tensor.cu) from int32 sums and row counts.
For +-11 ratings co-rated over a whole row of K, Mi = K^2 sum (x - mean)^2 reaches 121 K^3, which leaves int64 from
K ~ 4.24e5 (1..5: 4 K^3, from ~1.32e6), and its partial terms (K^2 Sxx, 2 K sa Sx) from ~3.4e5 (1..5: ~1.1e6).  Each
fixture below is item-based: every user rates every item, so every pair of items is co-rated over all K users.

The int32 accumulators: with m the largest |rating| and n2 the second-longest left row, a Fit whose sums can leave
int32 (4 m^2 n2 for MSD, m^2 n2 for Cosine and Pearson `sums`) must not run on the tensor path: an explicit
simPath="tensor" is refused, `auto` takes the exact stream path.  Two rows co-rated by every user, one +11 and one
-11 (sum (x - y)^2 = 484 n), sit at the MSD limit: n = 4,436,949 is the largest exact tensor Fit, 4,436,950 the first
refused one.

The regime test needs no GPU; the others print the largest ulp distance seen and their wall time."""
import time

import numpy as np
import pytest

import exact_sums as ex
from conftest import bits_equal

INT32_MAX = (1 << 31) - 1
RS_ERR_UNSUPPORTED = -3
MSD_EDGE = 4_436_949            # the largest n with 4 * 121 * n <= 2^31 - 1
COS_EDGE = 17_747_798           # the largest n with 121 * n <= 2^31 - 1


# ---------------------------------------------------------------------------------------------------------
# long-row fixtures: (items x K users, every cell rated)
# ---------------------------------------------------------------------------------------------------------
def _balanced(rng, k, lo, hi):
    """A row of k ratings, half lo and half hi, in random order."""
    return rng.permutation(np.repeat(np.array([lo, hi], dtype=np.float64), k // 2))


def _pm11_mixed(k, seed):
    """+-11: a balanced row, its copy (Pearson exactly 1) and negation (exactly -1), a random row, and two rows that
    are 90 % +11 (sa = 0.8 * 11 K: Mi = 0.36 * 121 K^3, whose partial terms still pass 121 K^3)."""
    rng = np.random.RandomState(seed)
    b = _balanced(rng, k, -11.0, 11.0)
    rows = [b, b.copy(), -b, rng.choice([-11.0, 11.0], k)]
    rows += [np.where(rng.uniform(size=k) < 0.9, 11.0, -11.0) for _ in range(2)]
    return np.stack(rows)


def _pm11_all_past(k, seed):
    """+-11: a balanced row, its copy, its negation and three random rows: every Mi past int64 at K = 6e5."""
    rng = np.random.RandomState(seed)
    b = _balanced(rng, k, -11.0, 11.0)
    return np.stack([b, b.copy(), -b] + [rng.choice([-11.0, 11.0], k) for _ in range(3)])


def _one_five(k, seed):
    """1 and 5 only, half each: a balanced row, its copy, its mirror 6 - x (exactly -1) and a random row."""
    rng = np.random.RandomState(seed)
    b = _balanced(rng, k, 1.0, 5.0)
    return np.stack([b, b.copy(), 6.0 - b, rng.choice([1.0, 5.0], k)])


# name -> (builder, K, what overflows int64 at the parent: "final" = some Mi, Ni or L itself (wrong there),
# "partial" = only partial terms (right there only by two's-complement wraparound), "none")
LONG = {"pm11_k450k": (_pm11_mixed, 450_000, {"final", "partial"}),
        "pm11_k600k": (_pm11_all_past, 600_000, {"final"}),
        "one_five_k1400k": (_one_five, 1_400_000, {"final"}),
        "one_five_k1300k": (_one_five, 1_300_000, {"partial"}),
        "pm11_k300k": (_pm11_mixed, 300_000, {"none"}),
        # the longest +-11 rows of the int64 epilogue: 4 * 121 * K^3 < 2^63 up to K = 267,104
        "pm11_k265k": (_pm11_mixed, 265_000, {"none"})}


def _long(name):
    build, k, _ = LONG[name]
    R = build(k, 0x10 + k)
    n_items = R.shape[0]
    left = np.repeat(np.arange(n_items, dtype=np.int32), k)
    right = np.tile(np.arange(k, dtype=np.int32), n_items)
    return left, right, R.ravel(), n_items, k


def _regimes(s):
    """For every off-diagonal pair: does Mi, Ni or L leave int64 ("final"), or only a partial term or partial sum of
    pearson_from_sums' int64 evaluation ("partial")?  Python ints, term by term as the parent evaluated them."""
    out = set()
    n_left = len(s.row_cnt)
    for a in range(n_left):
        for b in range(n_left):
            if a == b:
                continue
            n, sx, sy, sxx, syy, sxy = (int(v) for v in s.six(a, b))
            ca, sa, cb, sb = int(s.row_cnt[a]), int(s.row_sum[a]), int(s.row_cnt[b]), int(s.row_sum[b])
            t_mi = [ca * ca, ca * ca * sxx, 2 * ca, 2 * ca * sa, 2 * ca * sa * sx, n * sa, n * sa * sa]
            t_ni = [cb * cb, cb * cb * syy, 2 * cb, 2 * cb * sb, 2 * cb * sb * sy, n * sb, n * sb * sb]
            t_l = [ca * cb, ca * cb * sxy, ca * sb, ca * sb * sx, cb * sa, cb * sa * sy, n * sa, n * sa * sb]
            mi = ca * ca * sxx - 2 * ca * sa * sx + n * sa * sa
            ni = cb * cb * syy - 2 * cb * sb * sy + n * sb * sb
            lv = ca * cb * sxy - ca * sb * sx - cb * sa * sy + n * sa * sb
            t_sums = [ca * ca * sxx - 2 * ca * sa * sx, cb * cb * syy - 2 * cb * sb * sy, ca * cb * sxy - ca * sb * sx,
                      ca * cb * sxy - ca * sb * sx - cb * sa * sy]
            fits = lambda v: -ex.TWO63 <= v < ex.TWO63
            if not all(fits(v) for v in (mi, ni, lv)):
                out.add("final")
            elif not all(fits(v) for v in t_mi + t_ni + t_l + t_sums):
                out.add("partial")
            else:
                out.add("none")
    return out


@pytest.mark.parametrize("name", sorted(LONG))
def test_long_fixtures_are_in_their_regime(name):
    left, right, r, n_left, k = _long(name)
    s = ex.Sums(left, right, r, n_left, k)
    assert (s.n[~np.eye(n_left, dtype=bool)] == k).all()              # every pair co-rated over the whole row
    want, got = LONG[name][2], _regimes(s)
    if want == {"none"}:
        assert got == {"none"}, got
    else:
        assert got - {"none"} == want, got
    if name == "pm11_k600k":
        assert got == {"final"}                                       # every pair


# ---------------------------------------------------------------------------------------------------------
# device
# ---------------------------------------------------------------------------------------------------------
def _rs():
    import recommend_sys_b200 as rs

    return rs


def _handle(sim, path, **extra):
    return _rs().core._Handle(sim=sim, sim_path=path, **extra)


def _path(h):
    return {v: k for k, v in _rs().core.RS_SIM_PATH.items()}[h.profile()["sim_path_used"]]


def _fit(h, left, right, r, n_left, n_right):
    h.fit(left, right, r, n_left, n_right, float(np.mean(r)))
    h.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(LONG))
def test_long_rows_tensor(name, monkeypatch):
    """Pearson `sums`, Cosine and MSD on the tensor path over long rows: the rules of exact_sums.check_ratio, and
    Cosine / MSD bit for bit the numpy evaluation.  Pearson's epilogue is int64 up to K = 267,104 (pm11_k265k,
    pm11_k300k is past it) and __int128 beyond; the __int128 one forced on the same rows gives the same bits."""
    t0 = time.perf_counter()
    left, right, r, n_left, k = _long(name)
    s = ex.Sums(left, right, r, n_left, k)
    L, Mi, Ni = s.pearson_terms()
    pearson = []
    for force in ("0", "1"):
        monkeypatch.setenv("RS_KNN_PEARSON_I128", force)
        h = _handle("pearson", "tensor", pearson_mode="sums")
        _fit(h, left, right, r, n_left, k)
        assert _path(h) == "tensor"
        pearson.append(h.sims_rows(0, n_left))
        h.close()
    monkeypatch.delenv("RS_KNN_PEARSON_I128")
    assert bits_equal(pearson[0], pearson[1])
    worst = ex.check_ratio(pearson[0], L, Mi, Ni, who=name)
    assert worst[1] >= 0                                              # the fixture reaches |L|, Mi, Ni >= 2^53
    h = _handle("cosine", "tensor")
    _fit(h, left, right, r, n_left, k)
    assert _path(h) == "tensor"
    cos = h.sims_rows(0, n_left)
    h.close()
    assert bits_equal(cos, ex.cosine(s))
    worst_cos = ex.check_ratio(cos, s.sxy, s.sxx, s.syy, who=name + " cosine")
    h = _handle("msd", "tensor")
    _fit(h, left, right, r, n_left, k)
    assert _path(h) == "tensor"
    msd = h.sims_rows(0, n_left)
    h.close()
    assert bits_equal(msd, ex.msd(s))
    off = ~np.eye(n_left, dtype=bool)
    worst_msd = float(ex.ulps(msd[off], ex.msd_exact(s)[off]).max())
    assert worst_msd <= ex.MAX_ULPS_SMALL
    print(f"\n{name}: pearson max ulps (<2^53, >=2^53) = {worst}, cosine {worst_cos}, msd {worst_msd:.3f}; "
          f"{time.perf_counter() - t0:.1f} s")


def _two_rows(a, b):
    """Left rows 0 and 1 rated by users 0 .. len-1 with the given ratings."""
    left = np.concatenate([np.zeros(len(a), np.int32), np.ones(len(b), np.int32)])
    right = np.concatenate([np.arange(len(a), dtype=np.int32), np.arange(len(b), dtype=np.int32)])
    return left, right, np.concatenate([a, b]), 2, max(len(a), len(b))


def _refused(sim, data, who, **extra):
    rs = _rs()
    h = _handle(sim, "tensor", **extra)
    with pytest.raises(rs.core.RsError) as e:
        _fit(h, *data)
    assert e.value.code == RS_ERR_UNSUPPORTED
    assert who in str(e.value) and "2^31-1" in str(e.value), str(e.value)
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pair", ["0", "1"])
def test_msd_largest_exact_tensor_fit(pair, monkeypatch):
    """n = 4,436,949: 4 * 121 * n is the largest value an MSD int32 reaches below 2^31; single-CTA and pair kernel."""
    monkeypatch.setenv("RS_KNN_TC_PAIR", pair)
    t0 = time.perf_counter()
    n = MSD_EDGE
    assert 484 * n <= INT32_MAX < 484 * (n + 1)
    data = _two_rows(np.full(n, 11.0), np.full(n, -11.0))
    h = _handle("msd", "tensor")
    _fit(h, *data)
    assert _path(h) == "tensor"
    got = h.sims_rows(0, 2)
    h.close()
    want = 1.0 / (np.float64(484 * n) / np.float64(n) + 1.0)
    assert want == 1.0 / 485.0
    assert np.isnan(got[0, 0]) and np.isnan(got[1, 1])
    assert got[0, 1] == want and got[1, 0] == want, got
    print(f"\nMSD tensor Fit at K = {n} (pair={pair}): {time.perf_counter() - t0:.1f} s")


@pytest.mark.gpu
def test_msd_past_the_limit():
    """n = 4,436,950: 4 m^2 n2 = 2^31 + 152; the tensor path is refused, `auto` runs the exact stream path."""
    n = MSD_EDGE + 1
    data = _two_rows(np.full(n, 11.0), np.full(n, -11.0))
    _refused("msd", data, "4 m^2 n2")
    h = _handle("msd", "auto")
    _fit(h, *data)
    assert _path(h) == "stream"
    got = h.sims_rows(0, 2)
    h.close()
    assert got[0, 1] == 1.0 / 485.0 and got[1, 0] == 1.0 / 485.0


@pytest.mark.gpu
def test_cosine_and_pearson_past_the_limit():
    """m^2 n2 > 2^31 - 1 (n2 = 17,747,799 for Cosine; 17,747,800 for Pearson, whose two balanced rows have the
    exact mean 0, so that the reference's float64 sums are exact): explicit tensor and rs_knn_cosums are refused,
    `auto` takes the stream path and is exact.  No tensor kernel runs."""
    t0 = time.perf_counter()
    rng = np.random.RandomState(0xC05)
    n = COS_EDGE + 1
    a, b = _balanced(rng, n + 1, -11.0, 11.0), _balanced(rng, n + 1, -11.0, 11.0)
    for sim, data, extra in (("cosine", _two_rows(a, b[:n]), {}),
                             ("pearson", _two_rows(a, b), {"pearson_mode": "sums"})):
        s = ex.Sums(*data)
        assert 121 * int(np.sort(s.row_cnt)[-2]) > INT32_MAX
        _refused(sim, data, "m^2 n2", **extra)
        h = _handle(sim, "auto", **extra)
        _fit(h, *data)
        assert _path(h) == "stream"
        got = h.sims_rows(0, 2)
        with pytest.raises(_rs().core.RsError) as e:
            h.cosums(0, 1)
        assert e.value.code == RS_ERR_UNSUPPORTED and "m^2 n1" in str(e.value)
        h.close()
        # Cosine; and Pearson with both means exactly 0: Sxy / (sqrt(Sxx) sqrt(Syy)) in the reference's operations
        assert (s.row_sum == 0).all() or sim == "cosine"
        assert bits_equal(got, ex.cosine(s)), (sim, got)
        L, Mi, Ni = s.pearson_terms() if sim == "pearson" else (s.sxy, s.sxx, s.syy)
        ex.check_ratio(got, L, Mi, Ni, who=sim)
    print(f"\nCosine / Pearson past the int32 limit: {time.perf_counter() - t0:.1f} s")


@pytest.mark.gpu
def test_slope_one_past_the_limit():
    """Slope One's epilogue forms Sx - Sy in int32, up to 2 m n2: one row all +11 and one all -11 over n2 = 97,612,894
    users give 22 n2 = 2^31 + 2, and the Fit is refused (Slope One has no other path).  No tensor kernel runs."""
    t0 = time.perf_counter()
    n = INT32_MAX // 22 + 1
    assert n == 97_612_894 and 22 * (n - 1) <= INT32_MAX < 22 * n
    data = _two_rows(np.full(n, 11.0), np.full(n, -11.0))
    _refused("slope_one", data, "2 m n2")
    print(f"\nSlope One past the int32 limit: {time.perf_counter() - t0:.1f} s")
