"""The integer rating class over its whole range, against the oracle.

A rating set whose values are all integers in [-11, 11] (-0.0 included) is the integer class (RS_CLASS_INT8,
csrc/prep.cu): it enables the int8 planes and kind::i8 MMAs of the tensor path (signed operands), the byte codes
rating + 12 (the integer row sums of the means, the popular-column table of the exact sparse Fit and its decode),
Slope One and rs_knn_cosums.  The MovieLens fixtures only hold ratings 1..5, where every plane is non-negative, every
Cosine is >= 0 and every byte code is >= 13, so a sign error in any of these would pass them.  The fixtures here are
built to hold what those cannot: negative and extreme ratings, negative Cosine (exact -1, +0 and +1 among them,
negative k-th neighbours), shapes at the tile and K-block edges, long rows with negative ratings as popular columns,
and the edges of the class itself.  The coverage test needs no GPU; the others hold the device to the oracle bit
for bit (Pearson `sums` to its documented tolerance)."""
import numpy as np
import pytest

from conftest import ROOT, bits_equal
from oracle import binding as ob

VALUES = np.concatenate([np.arange(-11.0, 12.0), [-0.0]])     # every integer of the class, and -0.0
N_EDGES = (127, 128, 129, 255, 256, 257)                      # rows of the compared side around the 128-row tiles
K_EDGES = (63, 64, 65, 127, 129, 255, 257)                    # columns around the 64-byte / 128-byte K blocks
SHAPES = ((127, 63), (128, 64), (129, 65), (255, 127), (256, 129), (257, 255), (129, 257))   # (users, items)
POP_MIN = 150
K_TOP = 40
RS_ERR_UNSUPPORTED = -3


# ---------------------------------------------------------------------------------------------------------
# fixtures (deterministic)
# ---------------------------------------------------------------------------------------------------------
def _skewed_mask(rng, n_users, n_items, nnz):
    """About nnz cells rated with a MovieLens-like spread: log-normal user activity times log-normal item popularity
    (a long tail of rarely rated ids, whose rows have few neighbours)."""
    w = np.outer(rng.lognormal(0.0, 2.0, n_users), rng.lognormal(0.0, 2.0, n_items))
    lo, hi = 0.0, 1.0 / w.min()
    for _ in range(60):                     # the scale at which the expected number of rated cells is nnz
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if np.minimum(1.0, w * mid).sum() < nnz else (lo, mid)
    mask = rng.uniform(size=w.shape) < np.minimum(1.0, w * lo)
    return _with_tail(rng, mask)


def _with_tail(rng, mask, n_tail=16):
    """`mask` with n_tail more users who rate one item each, and n_tail more items rated by one user each, an item
    (user) of 48 to 80 ratings: on either side such a row's Cosine is +-1 against the 48 to 80 rows it shares that
    entry with, about half of them -1, so its k-th best at k = 40 is negative."""
    nu, ni = mask.shape
    out = np.zeros((nu + n_tail, ni + n_tail), dtype=bool)
    out[:nu, :ni] = mask
    items = np.flatnonzero((mask.sum(axis=0) >= 48) & (mask.sum(axis=0) <= 80))
    users = np.flatnonzero((mask.sum(axis=1) >= 48) & (mask.sum(axis=1) <= 80))
    out[nu + np.arange(n_tail), rng.choice(items, n_tail)] = True
    out[rng.choice(users, n_tail), ni + np.arange(n_tail)] = True
    return out


def _triples(rng, mask, values):
    """(users, items, ratings) of the cells of `mask` in a shuffled dataset order, values drawn from `values`."""
    uu, ii = np.nonzero(mask)
    order = rng.permutation(len(uu))
    return uu[order].astype(np.int64), ii[order].astype(np.int64), values[rng.randint(0, len(values), len(uu))]


def _uniform_parts(seed=0x1A7):
    rng = np.random.RandomState(seed)
    u, i, r = _triples(rng, _skewed_mask(rng, 1000, 600, 44_000), VALUES)
    return rng, u, i, r


def make_uniform():
    """Every value of [-11, 11] and -0.0 equally likely: ~950 users x ~600 items with ~40k training ratings, the
    last 4000 rated cells held out as test pairs.  Returns (u, i, r, test_u, test_i)."""
    _, u, i, r = _uniform_parts()
    return u[:-4000], i[:-4000], r[:-4000], u[-4000:], i[-4000:]


def make_extremes(seed=0xE11):
    """Only +-11 (every X^2 cell is 121): 600 x 400, plus three users who rate every item and two items every user
    rates, so that some pairs are co-rated over a whole side (Sxx = Syy = 121 K)."""
    rng = np.random.RandomState(seed)
    mask = _skewed_mask(rng, 600, 400, 20_000)
    mask[[5, 300, 599], :] = True
    mask[:, [7, 200]] = True
    return _triples(rng, mask, np.array([-11.0, 11.0]))


def make_like_dislike(seed=0x11D):
    """Only +-1: Cosine is exactly +-1 on one co-rated item, exactly 0 on balanced pairs; many ties at the k-th
    neighbour and rows whose k-th best is negative."""
    rng = np.random.RandomState(seed)
    return _triples(rng, _skewed_mask(rng, 600, 400, 12_000), np.array([-1.0, 1.0]))


def make_shape(n_users, n_items, seed=0x5A9E):
    """A quarter-filled n_users x n_items set in which every user and every item is rated (so the inner counts are
    exactly n_users and n_items), values as in make_uniform."""
    rng = np.random.RandomState(seed + 1000 * n_users + n_items)
    mask = rng.uniform(size=(n_users, n_items)) < 0.25
    mask[np.arange(n_users), np.arange(n_users) % n_items] = True
    mask[np.arange(n_items) % n_users, np.arange(n_items)] = True
    return _triples(rng, mask, VALUES)


def make_popular(seed=0x909):
    """make_uniform's training set plus six users and six items long enough to be popular columns at RS_KNN_POP_MIN
    = 150 (~360 and ~420 ratings), their ratings drawn from [-11, 11] with -11 and 11 twice as likely."""
    rng = np.random.RandomState(seed)
    u, i, r = make_uniform()[:3]
    mask = np.zeros((u.max() + 1, i.max() + 1), dtype=bool)
    mask[u, i] = True
    heavy = np.zeros_like(mask)
    heavy[[3, 250, 500, 750, 998, 999], :] = rng.uniform(size=(6, mask.shape[1])) < 0.6
    heavy[:, [1, 150, 300, 450, 598, 599]] |= rng.uniform(size=(mask.shape[0], 6)) < 0.42
    heavy &= ~mask
    hu, hi, hr = _triples(rng, heavy, np.concatenate([VALUES, [-11.0, 11.0]]))
    return np.concatenate([u, hu]), np.concatenate([i, hi]), np.concatenate([r, hr])


FIXTURES = {"uniform": lambda: make_uniform()[:3], "extremes": make_extremes, "like_dislike": make_like_dislike}


def _left(u, i, user_based):
    return (u, i) if user_based else (i, u)


_ORACLE = {}


def oracle(name, data, sim, user_based, knn_type="basic", k=K_TOP):
    """The oracle fitted on a fixture, one per (fixture, sim, orientation, type, k) and module."""
    key = (name, sim, user_based, knn_type, k)
    if key not in _ORACLE:
        u, i, r = data[:3]
        _ORACLE[key] = ob.KNN(sim=sim, knn_type=knn_type, user_based=user_based, k=k, n_jobs=8,
                              tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    return _ORACLE[key]


def _all_fixtures():
    """(name, data) of fixtures 1-4: the three value sets and every shape set."""
    out = [(name, make()) for name, make in FIXTURES.items()]
    return out + [(f"shape{nu}x{ni}", make_shape(nu, ni)) for nu, ni in SHAPES]


# ---------------------------------------------------------------------------------------------------------
# what the fixtures reach (oracle only, no GPU)
# ---------------------------------------------------------------------------------------------------------
def test_fixtures_reach_the_signed_range():
    if not (ROOT / "oracle" / "libknn_oracle.so").exists():
        pytest.skip("the oracle library is not built")
    u, i, r = make_uniform()[:3]
    assert set(np.unique(r).tolist()) == set(range(-11, 12))
    assert ((r == 0) & np.signbit(r)).sum() > 100 and ((r == 0) & ~np.signbit(r)).sum() > 100
    ex = make_extremes()
    assert set(np.unique(ex[2]).tolist()) == {-11.0, 11.0}
    assert np.bincount(ex[0]).max() == len(np.unique(ex[1]))               # users who rate every item
    assert np.bincount(ex[1]).max() == len(np.unique(ex[0]))               # items every user rates
    for name, data in (("uniform", (u, i, r)), ("like_dislike", make_like_dislike())):
        for user_based in (True, False):
            ref = oracle(name, data, "cosine", user_based)
            S = ref.sims(copy=False)
            fin = S[~np.isnan(S)]
            assert (fin < 0).sum() > 1000, (name, user_based)
            assert ((fin == 0) & ~np.signbit(fin)).sum() > 10, (name, user_based)
            assert (fin == 1.0).sum() > 100 and (fin == -1.0).sum() > 100, (name, user_based)
            _, ws = ref.topk(K_TOP)
            kth = ws[:, K_TOP - 1]
            assert (kth < 0).sum() >= 5, (name, user_based, (kth < 0).sum())       # negative k-th best
    pu, pi, pr = make_popular()
    for user_based in (True, False):
        left = _left(pu, pi, user_based)[0]
        lens = np.bincount(left)
        long_rows = np.flatnonzero(lens >= POP_MIN)
        assert len(long_rows) >= 2, user_based
        in_long = np.isin(left, long_rows)
        assert (pr[in_long] < 0).sum() > 100 and (pr[in_long] == -11).any() and (pr[in_long] == 11).any()
    n_seen, k_seen = set(), set()
    for nu, ni in SHAPES:
        su, si, _ = make_shape(nu, ni)
        assert len(np.unique(su)) == nu and len(np.unique(si)) == ni
        n_seen.add(nu)
        k_seen.add(ni)
    assert set(N_EDGES) <= n_seen and set(K_EDGES) <= k_seen


# ---------------------------------------------------------------------------------------------------------
# the tensor path's integer limits (host only)
# ---------------------------------------------------------------------------------------------------------
INT32_MAX = (1 << 31) - 1


def tensor_max_n2(sim, m):
    """The longest second-longest left row n2 whose co-rated sums the tensor path's int32 accumulators hold, for ratings
    of |x| <= m (tensor_eligible, csrc/api.cu): 4 m^2 n2 (MSD's Sum (x - y)^2), m^2 n2 (Cosine, Pearson `sums`:
    Sxx, Syy, |Sxy|), 2 m n2 (Slope One: its epilogue forms Sx - Sy)."""
    return INT32_MAX // {"msd": 4 * m * m, "cosine": m * m, "pearson": m * m, "slope_one": 2 * m}[sim]


def test_tensor_int32_limits():
    """+-11: MSD up to n2 = 4,436,949, Cosine and Pearson `sums` up to 17,747,798, Slope One up to 97,612,893.  Pearson
    forms Mi, Ni and L in int64 while 4 m^2 n1^3 < 2^63 (rows of up to 267,104 ratings of +-11), else in __int128:
    with every sum below 2^31 (and its row sums, |sa| <= m n1 < 2^31) the largest partial term n sa^2 stays below
    2^93.  Every workload of bench.py (ratings 1..5) is inside the limits of its
    similarity on the longest possible rows (a left row is at most as long as the other side has ids)."""
    import bench

    assert tensor_max_n2("msd", 11) == 4_436_949 and tensor_max_n2("cosine", 11) == 17_747_798
    assert tensor_max_n2("slope_one", 11) == 97_612_893
    assert 4 * 121 * 4_436_950 > INT32_MAX and 121 * 17_747_799 > INT32_MAX and 22 * 97_612_894 > INT32_MAX
    # Slope One's |Sx - Sy| reaches 2 m n2: one row all +11, the other all -11
    assert 11 * 97_612_894 - (-11) * 97_612_894 > INT32_MAX >= 11 * 97_612_893 - (-11) * 97_612_893
    # the int64 Pearson epilogue: every term is at most 4 m^2 n1^3
    assert 4 * 121 * 267_104 ** 3 < 1 << 63 <= 4 * 121 * 267_105 ** 3
    assert INT32_MAX * INT32_MAX ** 2 < 1 << 93
    for name, (users, items, *_rest, user_based, _k) in bench.WORKLOADS.items():
        longest = items if user_based else users
        for sim in ("msd", "cosine", "pearson", "slope_one"):
            assert longest <= tensor_max_n2(sim, 5), (name, sim)
    # with ratings of +-11 the Netflix item shape (480,189 users) would still be inside every limit
    assert bench.WORKLOADS["netflix_item_cosine_k50"][0] <= tensor_max_n2("msd", 11)


# ---------------------------------------------------------------------------------------------------------
# device against the oracle
# ---------------------------------------------------------------------------------------------------------
def _rs():
    import recommend_sys_b200 as rs

    return rs


def _sim(name):
    rs = _rs()
    return {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson}[name]


def _fit(data, sim, user_based, ctor="basic", **extra):
    rs = _rs()
    u, i, r = data[:3]
    ctors = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore}
    est = ctors[ctor](rs.Parameters(dict({"sim": _sim(sim), "userBased": user_based, "k": K_TOP}, **extra)))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    return est


def _path(est):
    rs = _rs()
    return {v: k for k, v in rs.core.RS_SIM_PATH.items()}[est.Profile()["sim_path_used"]]


VARIANTS = {"single": {"RS_KNN_TC_PAIR": "0"},
            "pair": {"RS_KNN_TC_PAIR": "1"}}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd"])
def test_tensor_sims_signed(sim, user_based, variant, monkeypatch):
    """Every tensor kernel variant on negative, extreme and +-1 ratings and at the tile / K-block edges."""
    for key, val in VARIANTS[variant].items():
        monkeypatch.setenv(key, val)
    for name, data in _all_fixtures():
        est = _fit(data, sim, user_based, simPath="tensor")
        assert _path(est) == "tensor"
        got = est.Sims
        assert np.isnan(np.diag(got)).all()
        assert bits_equal(got, oracle(name, data, sim, user_based).sims(copy=False)), name
        assert bits_equal(got, got.T), name
        est.Close()


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd"])
def test_tensor_equals_stream(sim, user_based):
    for name, data in _all_fixtures():
        a = _fit(data, sim, user_based, simPath="tensor")
        b = _fit(data, sim, user_based, simPath="stream")
        assert _path(b) == "stream"
        assert bits_equal(a.Sims, b.Sims), name
        a.Close()
        b.Close()


def _union(parts):
    import torch

    from recommend_sys_b200.shard import union_topk_device

    all_i = torch.from_numpy(np.stack([a for a, _ in parts])).cuda()
    all_s = torch.from_numpy(np.stack([b for _, b in parts])).cuda()
    uni_i, uni_s = union_topk_device(all_i, all_s)
    torch.cuda.synchronize()
    return uni_i.cpu().numpy(), uni_s.cpu().numpy()


SCHEDULES = {"fused_cap1792": {"RS_KNN_TOPK_FUSED": "1", "RS_KNN_TOPK_CAP": "1792"},
             "fused_cap96": {"RS_KNN_TOPK_FUSED": "1", "RS_KNN_TOPK_CAP": "96"},
             "symmetric_slabs": {"RS_KNN_TOPK_FUSED": "0", "RS_KNN_SLAB_ROWS": "128"},
             "row_slabs": {"RS_KNN_TOPK_FUSED": "0", "RS_KNN_SLAB_ROWS": "128"}}


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", sorted(SCHEDULES))
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("name", ["uniform", "like_dislike"])
def test_topk_schedules_negative_neighbours(name, user_based, schedule, monkeypatch):
    """Cosine top-k lists of the top-k-only store on the tensor path against the stream path's matrix TopK (itself
    the oracle's): the fused epilogue (every row's threshold starts at "not full", negative keys must pass it; a
    candidate buffer of 96 forces the overflow path), symmetric slabs and full-row slabs.  One shard, and three
    united, are the same lists."""
    data = FIXTURES[name]()
    full = _fit(data, "cosine", user_based, simPath="stream")
    want_i, want_s = full.TopK(K_TOP)
    full.Close()
    ref_i, ref_s = oracle(name, data, "cosine", user_based).topk(K_TOP)
    assert np.array_equal(want_i, ref_i) and bits_equal(want_s, ref_s)
    assert (want_s[:, K_TOP - 1] < 0).any()
    for key, val in SCHEDULES[schedule].items():
        monkeypatch.setenv(key, val)
    base = {"simPath": "tensor", "store": "topk", "topk": K_TOP}
    shard_counts = (None,) if schedule == "row_slabs" else (1, 3)
    for count in shard_counts:
        if count is None:
            est = _fit(data, "cosine", user_based, **base)
            got = est.TopK(K_TOP)
            est.Close()
        else:
            parts = []
            for rank in range(count):
                est = _fit(data, "cosine", user_based, shardCount=count, shardIndex=rank, **base)
                assert _path(est) == "tensor"
                parts.append(est.TopK(K_TOP))
                est.Close()
            got = parts[0] if count == 1 else _union(parts)
        assert np.array_equal(got[0], want_i), count
        assert bits_equal(got[1], want_s), count


def _exact(data, user_based):
    """The exact sums of a fixture (tests/exact_sums.py) over the inner ids the device sees, and Pearson's (L, Mi, Ni)."""
    import exact_sums as ex

    rs = _rs()
    ts = rs.NewTrainSet(rs.NewRawSet(*data[:3]))
    left, right = _left(ts.innerUsers, ts.innerItems, user_based)
    n_left, n_right = (ts.UserCount, ts.ItemCount) if user_based else (ts.ItemCount, ts.UserCount)
    s = ex.Sums(left, right, ts.Ratings, n_left, n_right)
    return s, s.pearson_terms()


# Pearson's tiles are 128 x 64 left rows with 128-byte K blocks: rows of the compared side around 64 and 192
PEARSON_SHAPES = ((63, 193), (64, 192), (65, 191), (191, 65), (192, 64), (193, 63))


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("name", ["uniform", "extremes", "shapes"])
def test_pearson_sums_signed(name, user_based):
    """Pearson `sums` within 1e-9 of the oracle's exact replay and, against the exact integers, with NaN exactly where
    Mi Ni == 0, +0.0 exactly where L == 0, bit-symmetric and within 4 ulps (6 past 2^53) of the exact value.  "shapes":
    the int-range shapes and Pearson's own tile edges."""
    import exact_sums as ex

    if name == "shapes":
        cases = [(f"shape{nu}x{ni}", make_shape(nu, ni)) for nu, ni in SHAPES + PEARSON_SHAPES]
    else:
        cases = [(name, FIXTURES[name]())]
    worst = [-1.0, -1.0]
    for case, data in cases:
        est = _fit(data, "pearson", user_based, simPath="tensor", pearsonMode="sums")
        assert _path(est) == "tensor"
        got, want = est.Sims, oracle(case, data, "pearson", user_based).sims(copy=False)
        assert np.array_equal(np.isnan(got), np.isnan(want)), case
        ok = ~np.isnan(want)
        err = np.abs(got[ok] - want[ok])
        assert (err <= 1e-9 * np.maximum(1.0, np.abs(want[ok]))).all(), (case, err.max())
        assert bits_equal(got, got.T), case
        _, (L, Mi, Ni) = _exact(data, user_based)
        w = ex.check_ratio(got, L, Mi, Ni, who=case)
        worst = [max(a, b) for a, b in zip(worst, w)]
        est.Close()
    print(f"\nPearson sums {name} user_based={user_based}: max ulps (<2^53, >=2^53) = {tuple(worst)}")


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
def test_pearson_sums_i128_epilogue(user_based, monkeypatch):
    """The __int128 instantiation of pearson_from_sums (the one Fits with rows past 267,104 ratings of +-11 run) forced
    on short rows gives the int64 one's bits: both form the same exact integers and round them the same way."""
    cases = [(name, FIXTURES[name]()) for name in ("uniform", "extremes")]
    cases += [(f"shape{nu}x{ni}", make_shape(nu, ni)) for nu, ni in PEARSON_SHAPES]
    for case, data in cases:
        got = []
        for force in ("0", "1"):
            monkeypatch.setenv("RS_KNN_PEARSON_I128", force)
            est = _fit(data, "pearson", user_based, simPath="tensor", pearsonMode="sums")
            assert _path(est) == "tensor"
            got.append(est.Sims)
            est.Close()
        assert bits_equal(got[0], got[1]), case


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
def test_pearson_sums_row_shards(user_based):
    """Contiguous row shards in `sums` mode (the non-mirrored tile list, row_begin > 0): each shard is its rows of the
    full-handle Fit bit for bit and meets the exact rules; aligned and unaligned boundaries."""
    import exact_sums as ex

    data = FIXTURES["uniform"]()
    full = _fit(data, "pearson", user_based, simPath="tensor", pearsonMode="sums")
    S = full.Sims
    full.Close()
    n = S.shape[0]
    _, (L, Mi, Ni) = _exact(data, user_based)
    for bounds in ((0, 384, n), (0, 100, 333, n), (0, 63, 65, n)):
        for b, e in zip(bounds[:-1], bounds[1:]):
            est = _fit(data, "pearson", user_based, simPath="tensor", pearsonMode="sums", rowBegin=b, rowEnd=e)
            assert _path(est) == "tensor"
            got = est.Sims
            est.Close()
            assert got.shape == (e - b, n)
            assert bits_equal(got, S[b:e]), (b, e)
            ex.check_ratio(got, L, Mi, Ni, row0=b, who=f"rows {b}:{e}")


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
def test_cosums_signed(user_based):
    """The six integer sums of rs_knn_cosums, negative Sx / Sy / Sxy included, for rows and columns at the tile
    edges."""
    data = FIXTURES["uniform"]()
    est = _fit(data, "msd", user_based, simPath="tensor")
    ref = oracle("uniform", data, "msd", user_based)
    n = est._h.n_left
    rng = np.random.RandomState(n)
    cols = np.unique(np.concatenate([rng.choice(n, 100), [0, 1, 63, 64, 65, 127, 128, 129, 255, 256, 257, n - 1]]))
    negative = 0
    for row0, nrows in ((0, 2), (126, 4), (254, 4), (n - 3, 3)):
        got = est._h.cosums(row0, nrows)
        assert got.shape == (nrows, n, 6)
        for r in range(nrows):
            for c in cols:
                want = ref.pair_sums(row0 + r, int(c))
                assert np.array_equal(got[r, c].astype(np.int64), want), (row0 + r, int(c))
                negative += int((want[[1, 2, 5]] < 0).any())
    assert negative > 50
    est.Close()


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("pop_min", ["0", str(POP_MIN)])
@pytest.mark.parametrize("tri", ["upper", "lower"])
@pytest.mark.parametrize("sim", ["cosine", "msd", "pearson"])
def test_popular_byte_table_signed(sim, tri, pop_min, user_based, monkeypatch):
    """The popular columns of the exact sparse Fit hold integer ratings as bytes rating + 12: negative ratings are
    the bytes below 12.  The set is the integer class (every rating an integer in [-11, 11]) and a full-matrix Fit
    with at least two rows of pop_min entries, which is what makes the table bytes."""
    monkeypatch.setenv("RS_KNN_STREAM_TRI", tri)
    monkeypatch.setenv("RS_KNN_STREAM_JC", "256")
    monkeypatch.setenv("RS_KNN_POP_MIN", pop_min)
    data = make_popular()
    r = data[2]
    assert (r == np.rint(r)).all() and (np.abs(r) <= 11).all()
    assert (np.bincount(_left(data[0], data[1], user_based)[0]) >= int(pop_min)).sum() >= 2
    est = _fit(data, sim, user_based, simPath="stream")
    assert _path(est) == "stream"
    got = est.Sims
    assert np.isnan(np.diag(got)).all()
    assert bits_equal(got, oracle("popular", data, sim, user_based).sims(copy=False))
    assert bits_equal(got, got.T)
    est.Close()


@pytest.mark.gpu
def test_popular_byte_table_cyclic_shards(monkeypatch):
    """Two cyclic row shards on one GPU, popular columns with negative bytes on both, mirrored: the full matrix."""
    monkeypatch.setenv("RS_KNN_POP_MIN", str(POP_MIN))
    data = make_popular()
    full = _fit(data, "pearson", False, "centered")
    want = full.Sims
    assert bits_equal(want, oracle("popular", data, "pearson", False).sims(copy=False))
    shards = [_fit(data, "pearson", False, "centered", shardCount=2, shardIndex=q) for q in range(2)]
    for est in shards:
        est._h.synchronize()
    for est in shards:
        est._h.peer_import_local([x._h for x in shards])
        est._h.mirror()
    for est in shards:
        assert bits_equal(est.Sims, want[est._h.owned_rows()])
        est.Close()
    full.Close()


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim,path", [("pearson", "stream"), ("msd", "stream"), ("cosine", "tensor")])
@pytest.mark.parametrize("ctor", ["centered", "zscore"])
def test_means_and_predict_signed(ctor, sim, path, user_based):
    """Means from the integer row sums (negative here), stddevs and held-out predictions."""
    u, i, r, tu, ti = make_uniform()
    est = _fit((u, i, r), sim, user_based, ctor, simPath=path)
    assert _path(est) == path
    ref = oracle("uniform", (u, i, r), sim, user_based, ctor)
    assert (ref.means() < 0).sum() > 100
    assert bits_equal(est.Means, ref.means())
    if ctor == "zscore":
        assert bits_equal(est.StdDevs, ref.stddevs())
    assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti, n_threads=8))
    est.Close()


@pytest.mark.gpu
@pytest.mark.parametrize("pair", ["0", "1"])
@pytest.mark.parametrize("name", ["uniform", "extremes"])
def test_slope_one_signed(name, pair, monkeypatch):
    """Slope One deviations up to 22 in magnitude, bit for bit (signed zeros too), and its predictions."""
    monkeypatch.setenv("RS_KNN_TC_PAIR", pair)
    rs = _rs()
    if name == "uniform":
        u, i, r, tu, ti = make_uniform()
    else:
        u, i, r = make_extremes()
        rng = np.random.RandomState(3)
        tu, ti = rng.randint(0, 600, 3000), rng.randint(0, 400, 3000)
    tu = np.concatenate([tu, [10 ** 9, tu[0], 10 ** 9]])                  # unknown user / item / both
    ti = np.concatenate([ti, [ti[0], 10 ** 9, 10 ** 9]])
    est = rs.NewSlopeOne(None)
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    ref = ob.SlopeOne().fit(ob.TrainSet(u, i, r))
    got, want = est.dev, ref.dev()
    assert np.abs(want).max() > 11
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti))
    est.Close()


@pytest.mark.gpu
def test_recommend_like_dislike_tensor():
    """Top-N recommendation from a tensor-path Cosine on +-1 ratings with k = 2: negative scores, and +-Inf where a
    +1 and a -1 neighbour cancel."""
    from recommend_ref import score_all
    from test_recommend_gpu import _check_handle

    data = make_like_dislike()
    u, i, r = data
    for user_based in (True, False):
        est = _fit(data, "cosine", user_based, simPath="tensor", k=2)
        assert _path(est) == "tensor"
        side = "left" if user_based else "right"
        q = np.arange(est._h.n_left if side == "left" else est._h.n_right)
        want = score_all(oracle("like_dislike", data, "cosine", user_based, k=2), u, i, user_based, side, q)
        got, _ = _check_handle(est._h, side, q, (1, 10, 512), want)
        fin = got[~np.isnan(got)]
        assert (fin < 0).any() and np.isposinf(fin).any() and np.isneginf(fin).any()
        est.Close()


@pytest.mark.gpu
@pytest.mark.parametrize("sim,ctor,user_based,path", [("cosine", "centered", True, "tensor"),
                                                       ("pearson", "zscore", False, "stream")])
def test_update_signed_delta(sim, ctor, user_based, path):
    """rs_knn_update on an integer-class model with ratings of the whole range (+-11 among them) = a refit."""
    from test_update_gpu import _same_model, _updated

    u, i, r, tu, ti = make_uniform()
    m = len(r) - 3000
    assert (r[m:] == 11).any() and (r[m:] == -11).any()
    got = _updated(u, i, r, m, sim, ctor, user_based, extra={"simPath": path})
    want = _fit((u, i, r), sim, user_based, ctor)
    _same_model(got, want, np.stack([tu, ti, np.zeros_like(tu)], axis=1))
    got.Close()
    want.Close()


# ---- the edges of the class: 11 and -11 are in, 12, -12 and 11.5 out, -0.0 in ----
def _dense_set(values, seed):
    rng = np.random.RandomState(seed)
    mask = rng.uniform(size=(200, 150)) < 0.5
    u, i, r = _triples(rng, mask, np.asarray(values, dtype=np.float64))
    return u, i, r


def _check_against_oracle(data, sim, path):
    est = _fit(data, sim, True, "centered", simPath=path)
    u, i, r = data
    ref = ob.KNN(sim=sim, knn_type="centered", user_based=True, k=K_TOP, n_jobs=8,
                 tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    assert bits_equal(est.Sims, ref.sims(copy=False))
    assert bits_equal(est.Means, ref.means())
    pu, pi = u[::7] + 1, i[::7]                              # pairs of neighbouring users, rated or not
    assert bits_equal(est.PredictBatch(pu, pi), ref.predict_batch(pu, pi))
    return est


@pytest.mark.gpu
@pytest.mark.parametrize("values", [np.arange(0.0, 12.0), np.arange(-11.0, 1.0)], ids=["to_11", "from_-11"])
def test_class_boundary(values):
    rs = _rs()
    data = _dense_set(values, 17)
    assert (np.abs(data[2]) == 11).any()
    for sim in ("cosine", "msd"):
        _check_against_oracle(data, sim, "tensor").Close()
        est = _fit(data, sim, True)
        assert _path(est) == "tensor"                      # auto takes the tensor path on this dense set
        est.Close()
    for bad in (12.0, -12.0, 11.5):
        u, i, r = data
        r = r.copy()
        r[len(r) // 2] = bad
        for sim in ("cosine", "msd"):
            est = _check_against_oracle((u, i, r), sim, "auto")
            assert _path(est) == "stream"                  # not the integer class any more
            est.Close()
            with pytest.raises(rs.core.RsError) as e:
                _fit((u, i, r), sim, True, simPath="tensor")
            assert e.value.code == RS_ERR_UNSUPPORTED
        with pytest.raises(rs.core.RsError) as e:
            rs.NewSlopeOne(None).Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
        assert e.value.code == RS_ERR_UNSUPPORTED


@pytest.mark.gpu
@pytest.mark.parametrize("call", ["host", "device"])
def test_update_outside_the_class_is_refused(call):
    """An integer-class model refuses 12, -12 and 11.5 and is left exactly as it was; +-11 are accepted."""
    from test_update_gpu import _raw_update, _raw_update_device, _same_snapshot, _snapshot

    run = _raw_update if call == "host" else _raw_update_device
    rs = _rs()
    u, i, r, tu, ti = make_uniform()
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    h = rs.core._Handle(sim="cosine", knn_type="zscore", sim_path="tensor")
    h.fit(ts.innerUsers, ts.innerItems, ts.Ratings, ts.UserCount, ts.ItemCount, ts.GlobalMean)
    nl, nr = h.n_left, h.n_right
    held = np.stack([tu, ti, np.zeros_like(tu)], axis=1)
    new = (ts.convert_users(tu) >= 0) & (ts.convert_items(ti) >= 0)
    lu, li = ts.convert_users(tu[new][:2]), ts.convert_items(ti[new][:2])     # pairs the model does not hold
    before = _snapshot(h, held)
    for bad in (12.0, -12.0, 11.5):
        assert run(h, lu, li, [4.0, bad], nl, nr) == RS_ERR_UNSUPPORTED, bad
        _same_snapshot(before, _snapshot(h, held))
    assert run(h, lu, li, [11.0, -11.0], nl, nr) == 0
    h.close()


@pytest.mark.gpu
def test_negative_zero_ratings():
    """-0.0 is an integer of the class: the set takes the tensor path under auto and matches the oracle fed the same
    -0.0 values; Slope One accepts it."""
    rs = _rs()
    data = _dense_set([-0.0, -0.0, 0.0, 1.0, -1.0, 2.0], 23)
    assert ((data[2] == 0) & np.signbit(data[2])).sum() > 1000
    for sim in ("cosine", "msd"):
        _check_against_oracle(data, sim, "tensor").Close()
        est = _check_against_oracle(data, sim, "auto")
        assert _path(est) == "tensor"
        est.Close()
    u, i, r = data
    est = rs.NewSlopeOne(None)
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    assert np.array_equal(est.dev.view(np.uint64), ob.SlopeOne().fit(ob.TrainSet(u, i, r)).dev().view(np.uint64))
    est.Close()
