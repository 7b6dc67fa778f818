"""Neighbour selection against the oracle in every regime of the selection code (csrc/predict.cu).

predict_select_kernel<R> picks the top min(k, valid) candidates of a prediction with a radix selection on
32-bit keys, falls back to exact 64-bit passes when one key32 value overfills the boundary bucket, takes
genuine ties in ascending id order and parks keys beyond its shared-memory stage in global memory; the
block top-k kernels (rows, symmetric slabs, fused epilogue, union) keep a running threshold once a row has
more candidates than their buffer.  The MovieLens folds reach most of these branches only by chance, so the
fixture here is designed: every prediction sees a chosen multiset of similarities over a chosen number of
candidates, and a host classifier (a restatement of the kernel's decisions) proves which branch each one
takes.  The coverage test needs no GPU; the others hold the device to the oracle bit for bit."""
import math

import numpy as np
import pytest

from conftest import bits_equal, split
from oracle import binding as ob

N_CAND = 3000                                  # candidate users; test item t is rated by the first SIZES[t]
SIZES = (1, 44, 45, 64, 65, 128, 129, 256, 257, 511, 512, 513, N_CAND)
K_SWEEP = (1, 44, 45, 104, 105, 200, 256)
MINK = 1
SCAP = 256                                     # default shared-memory stage of the predict kernel (keys / warp)
CAND0 = 10_000                                 # raw id of candidate 0; left rows are raw users 0 .. M-1
TEST0 = 100_000                                # raw id of test item 0


def cap_of(k):
    """Register capacity CAP = 32 * R of the predict kernel for this k (rs_predict_launch)."""
    return 32 * (2 if k <= 44 else 4 if k <= 104 else 8)


def _msd_patterns(rng):
    """Left row m rates pivot item m with 0.0; candidate c rates it with delta -> S = 1 / (delta^2 + 1).
    None = the candidate does not rate the pivot (S is NaN)."""
    c = np.arange(N_CAND, dtype=np.float64)
    ci = np.arange(N_CAND)
    nan = np.full(N_CAND, np.nan)
    collide = 1.0 + c * 2.0 ** -40             # S just below 0.5: one key32 value, distinct key64
    p = {
        "tie_all": np.zeros(N_CAND),                                       # S = 1.0 everywhere
        "tie_levels": np.array([0.0, 0.5, 1.0, 2.0, 3.0])[ci % 5],
        "tie_levels_random": rng.randint(0, 4, N_CAND) * 0.5,
        "tie_thirds": np.where(ci % 3 == 0, 0.0, nan),
        "collide": collide,
        "collide_sevenths": np.where(ci % 7 == 0, collide, nan),
        "collide_under_few": np.where(ci % 16 == 0, rng.uniform(0.0, 0.9, N_CAND), collide),
        "collide_under_many": np.where(ci % 3 == 0, rng.uniform(0.0, 0.9, N_CAND), collide),
        "spread": 2.0 ** (ci % 24) * (1.0 + rng.uniform(0.0, 1.0, N_CAND)),
        "spread_ties": 2.0 ** (ci % 20),
        "spread_collide": np.where(ci % 2 == 0, 2.0 ** (ci % 24) * 3.0, collide),
        "random": rng.uniform(0.0, 3.0, N_CAND),
        "random_halves": np.where(ci % 2 == 0, rng.uniform(0.0, 3.0, N_CAND), nan),
        "half_ones": np.where(ci % 2 == 0, 0.0, rng.uniform(0.1, 3.0, N_CAND)),
        "every_50": np.where(ci % 50 == 0, rng.uniform(0.0, 3.0, N_CAND), nan),
        "one_rater": np.where(ci == 0, 0.5, nan),                          # valid = mink
        "two_raters": np.where((ci == 0) | (ci == 300), 0.5, nan),         # valid = mink + 1 past 300 candidates
        "late_raters": np.where((ci == 2000) | (ci == 2001), 1.0, nan),    # valid = 0 below 2000 candidates
    }
    return p


def _cos_patterns(rng):
    """Left row m rates its two pivots with 1, 1; candidate c rates them (a, b) -> signed Cosine.  NaN in a
    column = that pivot is not rated (one rated pivot gives exactly +-1)."""
    ci = np.arange(N_CAND)
    nan = np.full(N_CAND, np.nan)
    th = rng.uniform(0.0, 2 * math.pi, N_CAND)
    sign = np.where(rng.randint(0, 2, N_CAND) == 0, -1.0, 1.0)
    mag = rng.uniform(0.5, 4.0, N_CAND)
    tiny = 2.0 ** -(ci % 30).astype(np.float64)
    p = {
        "c_tie_all": (np.full(N_CAND, math.cos(0.3)), np.full(N_CAND, math.sin(0.3))),
        "c_random": (np.cos(th), np.sin(th)),
        "c_ones": (sign * mag, nan),                                       # exactly +1 / -1
        "c_ones_random": (np.where(ci % 2 == 0, sign * mag, np.cos(th)), np.where(ci % 2 == 0, nan, np.sin(th))),
        "c_zeros": (np.array([1.0, 1.0, -1.0, 2.0])[ci % 4], np.array([-1.0, 1.0, -1.0, -2.0])[ci % 4]),
        "c_signed_spread": (np.ones(N_CAND), -1.0 + sign * tiny),          # +-2^-j / 2: many binades, both signs
        "c_collide_neg": (-np.ones(N_CAND), ci * 2.0 ** -40),               # -(1 - c 2^-40) / sqrt 2
        "c_collide_neg_few": (np.where(ci % 9 == 0, np.cos(th), -1.0), np.where(ci % 9 == 0, np.sin(th), ci * 2.0 ** -40)),
        "c_sparse": (np.where(ci % 40 == 0, np.cos(th), nan), np.where(ci % 40 == 0, np.sin(th), nan)),
        "c_two_raters": (np.where((ci == 5) | (ci == 400), -1.0, nan), np.where((ci == 5) | (ci == 400), 0.25, nan)),
    }
    return p


def make_fixture(kind, seed=0x5E1EC7):
    """(users, items, ratings, left raw ids, test item raw ids) of the designed data set; kind 'msd' or 'cosine'.

    Users: left rows 0 .. M-1 first, then the candidates in order, so that inner ids ascend with the
    candidate index and the canonical tie rule (ascending inner id) prefers earlier candidates."""
    rng = np.random.RandomState(seed)
    pats = _msd_patterns(rng) if kind == "msd" else _cos_patterns(rng)
    names = sorted(pats)
    m_rows = len(names)
    us, its, rs_ = [], [], []

    def add(u, i, r):
        us.append(np.asarray(u, dtype=np.int64))
        its.append(np.asarray(i, dtype=np.int64))
        rs_.append(np.asarray(r, dtype=np.float64))

    # left rows: one rating per pivot
    for m, name in enumerate(names):
        if kind == "msd":
            add([m], [2 * m], [0.0])
        else:
            add([m, m], [2 * m, 2 * m + 1], [1.0, 1.0])
    # candidates in ascending order: pivots of every pattern, then the test items
    test_r = 1.0 + rng.randint(0, 9, (len(SIZES), N_CAND)) * 0.5        # 1.0 .. 5.0 in half steps
    for c in range(N_CAND):
        uu, ii, rr = [], [], []
        for m, name in enumerate(names):
            if kind == "msd":
                d = pats[name][c]
                if not np.isnan(d):
                    uu.append(CAND0 + c); ii.append(2 * m); rr.append(d)
            else:
                a, b = pats[name][0][c], pats[name][1][c]
                for col, v in ((0, a), (1, b)):
                    if not np.isnan(v):
                        uu.append(CAND0 + c); ii.append(2 * m + col); rr.append(v)
        for t, n_t in enumerate(SIZES):
            if c < n_t:
                uu.append(CAND0 + c); ii.append(TEST0 + t); rr.append(test_r[t, c])
        add(uu, ii, rr)
    u, i, r = np.concatenate(us), np.concatenate(its), np.concatenate(rs_)
    return u, i, r, np.arange(m_rows, dtype=np.int64), TEST0 + np.arange(len(SIZES), dtype=np.int64)


def sim_keys(s):
    """rs_sim_key of float64 values (after s + 0.0), 0 for NaN; and the top 32 bits of it."""
    s = np.asarray(s, dtype=np.float64) + 0.0
    b = s.view(np.uint64)
    key = np.where(b >> np.uint64(63), ~b, b | np.uint64(1 << 63))
    key = np.where(np.isnan(s), np.uint64(0), key).astype(np.uint64)
    return key, (key >> np.uint64(32)).astype(np.uint64)


REGIMES = ("mink", "direct", "radix32", "fallback64", "tie_take", "below_top_binade", "spill32", "spill64")


def classify(row_sims, k, min_k=MINK, scap=SCAP):
    """Which branches of predict_select_kernel<R> one prediction takes.  row_sims: the similarities of the
    prediction's candidates in candidate (= inner id) order, NaN = not a neighbour."""
    cnt = len(row_sims)
    key, k32 = sim_keys(row_sims)
    key, k32 = key[key != 0], k32[key != 0]
    valid = len(key)
    if valid <= min_k:
        return {"mink"}
    cap = cap_of(k)
    num = min(k, valid)
    out = set()
    if cnt > 2 * scap:
        out.add("spill32")
    if valid <= cap:
        out.add("direct")
        return out
    t64 = np.sort(key)[::-1][num - 1]
    t32 = t64 >> np.uint64(32)
    a32, b32 = int((k32 > t32).sum()), int((k32 == t32).sum())
    top32 = int(k32.max())
    if int((k32 >= np.uint64(max(top32 - (1 << 20), 0))).sum()) < num:
        out.add("below_top_binade")
    if a32 + b32 <= cap:
        out.add("radix32")
        return out
    out.add("fallback64")
    if cnt > scap:
        out.add("spill64")
    a64, b64 = int((key > t64).sum()), int((key == t64).sum())
    if a64 + b64 > cap:
        out.add("tie_take")
    return out


def regime_table(S, left_inner, k_values):
    """counts[R][regime] over every (left row, test item) prediction at the given k values."""
    counts = {r: dict.fromkeys(REGIMES, 0) for r in (2, 4, 8)}
    for k in k_values:
        r = cap_of(k) // 32
        for m in left_inner:
            for n_t in SIZES:
                # test item t is rated by candidates 0 .. n_t - 1 = inner users M .. M + n_t - 1
                for reg in classify(S[m, len(left_inner):len(left_inner) + n_t], k):
                    counts[r][reg] += 1
    return counts


def _ref(data, kind, knn_type, k):
    u, i, r = data[:3]
    return ob.KNN(sim="msd" if kind == "msd" else "cosine", knn_type=knn_type, user_based=True, k=k, min_k=MINK,
                  n_jobs=8, tie_policy="canonical").fit(ob.TrainSet(u, i, r))


# ---------------------------------------------------------------------------------------------------------
# coverage of the designed fixture (host only)
# ---------------------------------------------------------------------------------------------------------
def test_fixture_reaches_every_selection_regime():
    """The classifier on the oracle's matrices: each fixture takes every regime at least 10 times for each
    register width."""
    for kind in ("msd", "cosine"):
        data = make_fixture(kind)
        u, i, r, left = data[:4]
        S = _ref(data, kind, "basic", 40).sims()
        iu, own = ob.TrainSet(u, i, r).inner_users(), u < len(left)             # the id layout the table relies on
        assert (iu[own] == u[own]).all() and (iu[~own] == u[~own] - CAND0 + len(left)).all()
        tab = regime_table(S, np.arange(len(left)), K_SWEEP)
        print(f"\n{kind}: " + " ".join(f"{x:>16}" for x in REGIMES))
        for R, row in tab.items():
            print(f"  R={R}: " + " ".join(f"{row[x]:>16}" for x in REGIMES))
        for R, row in tab.items():
            for x in REGIMES:
                assert row[x] >= 10, (kind, R, x, row)
        if kind == "cosine":
            fin = S[:len(left)][~np.isnan(S[:len(left)])]
            assert (fin < 0).sum() > 1000 and (fin == 0).sum() > 100       # signed values and zeros


# ---------------------------------------------------------------------------------------------------------
# device against the oracle
# ---------------------------------------------------------------------------------------------------------
def _rs():
    import recommend_sys_b200 as rs

    return rs


def _device_fit(kind, knn_type, **extra):
    rs = _rs()
    u, i, r, left, items = make_fixture(kind)
    params = {"sim": rs.MSD if kind == "msd" else rs.Cosine, "userBased": True, "k": 40, "mink": MINK,
              "simPath": "stream"}
    params.update(extra)
    ctor = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean}[knn_type]
    est = ctor(rs.Parameters(params))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    pu, pi = np.repeat(left, len(items)), np.tile(items, len(left))     # every (left row, test item) pair
    return est, (u, i, r, left, items), (pu, pi)


def _set_scap(monkeypatch, scap):
    if scap is None:
        monkeypatch.delenv("RS_KNN_PRED_SCAP", raising=False)
    else:
        monkeypatch.setenv("RS_KNN_PRED_SCAP", scap)


@pytest.mark.gpu
@pytest.mark.parametrize("knn_type", ["basic", "centered"])
@pytest.mark.parametrize("kind", ["msd", "cosine"])
def test_predict_sweep_every_k_and_stage(kind, knn_type, monkeypatch):
    """One fitted handle, k walked across both register-width switches up to the ABI maximum with
    rs_knn_set_k, under four shared-memory stage sizes (0 and 32: every key spills; 2048: none does)."""
    est, data, (pu, pi) = _device_fit(kind, knn_type)
    assert bits_equal(est.Sims, _ref(data, kind, knn_type, 40).sims())
    for k in K_SWEEP:
        want = _ref(data, kind, knn_type, k).predict_batch(pu, pi)
        for scap in (None, "0", "32", "2048"):
            _set_scap(monkeypatch, scap)
            est.Params["k"] = k
            got = est.PredictBatch(pu, pi)
            assert bits_equal(got, want), (k, scap, np.flatnonzero(~np.isclose(got, want, equal_nan=True))[:10])
    est.Close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["msd", "cosine"])
def test_neighbour_lists_every_k(kind, monkeypatch):
    """The neighbours Predict used, in accumulation order: ids and similarities bit for bit."""
    est, data, (pu, pi) = _device_fit(kind, "basic")
    S = _ref(data, kind, "basic", 40).sims()
    m_rows = len(data[3])
    for k in K_SWEEP:
        ref = _ref(data, kind, "basic", k)
        est.Params["k"] = k
        est.PredictBatch(pu[:1], pi[:1])                        # applies k to the handle (rs_knn_set_k)
        for scap in (None, "0"):
            _set_scap(monkeypatch, scap)
            for x, (uu, ii) in enumerate(zip(pu, pi)):
                gi, gs = est.Neighbors(int(uu), int(ii))
                n_t = SIZES[x % len(SIZES)]
                if "mink" in classify(S[x // len(SIZES), m_rows:m_rows + n_t], k):
                    assert len(gi) == 0
                    continue
                wi, ws = ref.predict_neighbors(int(uu), int(ii))
                assert len(wi) == min(k, np.count_nonzero(~np.isnan(S[x // len(SIZES), m_rows:m_rows + n_t])))
                assert np.array_equal(gi.astype(np.int64), wi), (k, scap, x)
                assert bits_equal(gs, ws), (k, scap, x)
    est.Close()


@pytest.mark.gpu
def test_k_beyond_the_predict_kernel_is_refused():
    rs = _rs()
    est, _, (pu, pi) = _device_fit("msd", "basic")
    est.Params["k"] = 257
    with pytest.raises(rs.core.RsError) as e:
        est.PredictBatch(pu, pi)
    assert e.value.code == -3                                 # RS_ERR_UNSUPPORTED
    est.Close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["msd", "cosine"])
def test_block_topk_every_k(kind):
    """topk_rows_kernel: the candidate rows hold ~3000 valid similarities (more than the 1792 that trigger
    the running threshold), the tie rows 3000 copies of one value; rows with fewer than k are padded."""
    rs = _rs()
    est, data, _ = _device_fit(kind, "basic")
    ref = _ref(data, kind, "basic", 40)
    valid = (~np.isnan(ref.sims(copy=False))).sum(axis=1)
    assert (valid > 1792).sum() > 2000 and (valid < 512).any()
    for k in (1, 40, 255, 256, 511, 512):
        gi, gs = est.TopK(k)
        wi, ws = ref.topk(k)
        assert np.array_equal(gi, wi), k
        assert bits_equal(gs, ws), k
    assert (wi == -1).any()                                   # padded rows (-1 / NaN) were compared
    if kind == "msd":
        assert (ws[:len(data[3])] == 1.0).sum() > 512         # the tie row fills its list with 1.0
    with pytest.raises(rs.core.RsError) as e:
        est.TopK(513)
    assert e.value.code == -3
    est.Close()


@pytest.mark.gpu
def test_slab_topk_at_the_buffer_limit(monkeypatch):
    """Symmetric slabs of 256 rows at k = 512 (one shard = the matrix-store lists); four shards united at
    n_lists * k = 2048, the union's buffer; one list more is refused."""
    import torch

    rs = _rs()
    from recommend_sys_b200.shard import union_topk_device

    monkeypatch.setenv("RS_KNN_SLAB_ROWS", "256")
    k = 512
    full, data, _ = _device_fit("msd", "basic")
    want_i, want_s = full.TopK(k)
    full.Close()
    one, _, _ = _device_fit("msd", "basic", store="topk", topk=k, shardCount=1)
    got_i, got_s = one.TopK(k)
    one.Close()
    assert np.array_equal(got_i, want_i) and bits_equal(got_s, want_s)
    parts = []
    for rank in range(4):
        p, _, _ = _device_fit("msd", "basic", store="topk", topk=k, shardCount=4, shardIndex=rank)
        parts.append(p.TopK(k))
        p.Close()
    all_i = torch.from_numpy(np.stack([a for a, _ in parts])).cuda()
    all_s = torch.from_numpy(np.stack([b for _, b in parts])).cuda()
    uni_i, uni_s = union_topk_device(all_i, all_s)
    torch.cuda.synchronize()
    assert np.array_equal(uni_i.cpu().numpy(), want_i) and bits_equal(uni_s.cpu().numpy(), want_s)
    with pytest.raises(rs.core.RsError) as e:
        union_topk_device(torch.cat([all_i, all_i[:1]]), torch.cat([all_s, all_s[:1]]))
    assert e.value.code == -3


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd"])
def test_fused_topk_at_the_buffer_limit(ml100k, sim, user_based, monkeypatch):
    """The fused epilogue at k = 256 with the default candidate capacity: 1792 + 256 = 2048 fills the merge
    buffer exactly; k = 257 is refused."""
    rs = _rs()
    monkeypatch.setenv("RS_KNN_TOPK_FUSED", "1")
    u, i, r = split(ml100k["u1_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    base = {"sim": rs.Cosine if sim == "cosine" else rs.MSD, "userBased": user_based}
    full = rs.NewKNN(rs.Parameters(dict(base, simPath="stream")))
    full.Fit(ts)
    want_i, want_s = full.TopK(256)
    full.Close()
    one = rs.NewKNN(rs.Parameters(dict(base, simPath="tensor", store="topk", topk=256, shardCount=1)))
    one.Fit(ts)
    got_i, got_s = one.TopK(256)
    one.Close()
    assert np.array_equal(got_i, want_i) and bits_equal(got_s, want_s)
    with pytest.raises(rs.core.RsError) as e:
        rs.NewKNN(rs.Parameters(dict(base, simPath="tensor", store="topk", topk=257, shardCount=1))).Fit(ts)
    assert e.value.code == -3


@pytest.mark.gpu
@pytest.mark.parametrize("user_based", [True, False])
def test_negative_zero_similarities_in_neighbour_lists(ml100k, user_based):
    """PearsonBaseline with shrinkage: a pair with one co-rated entry and residuals of opposite signs is
    exactly -0.0.  Lists order +-0 as equal (ties by id) and report the exact similarity."""
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    base = {"sim": rs.PearsonBaseline, "userBased": user_based, "shrinkage": 100.0}
    est = rs.NewKNNBaseLine(rs.Parameters(base))
    est.Fit(ts)
    ref = ob.KNN(sim="pearson_baseline", knn_type="baseline", user_based=user_based, n_jobs=8,
                 shrinkage=100.0).fit(ob.TrainSet(u, i, r))
    S = ref.sims(copy=False)
    assert ((S == 0) & np.signbit(S)).sum() > 10_000
    assert bits_equal(est.Sims, S)
    wi, ws = ref.topk(512)
    assert ((ws == 0) & np.signbit(ws)).sum() > 10_000
    gi, gs = est.TopK(512)
    assert np.array_equal(gi, wi) and bits_equal(gs, ws)
    slab = rs.NewKNNBaseLine(rs.Parameters(dict(base, store="topk", topk=512, shardCount=1)))
    slab.Fit(ts)
    si, ss = slab.TopK(512)
    slab.Close()
    assert np.array_equal(si, wi) and bits_equal(ss, ws)
    tu, ti, _ = split(ml100k["u1_test"])
    neg0 = 0
    for x in range(0, len(tu), 7):
        gi, gs = est.Neighbors(int(tu[x]), int(ti[x]))
        wi, ws = ref.predict_neighbors(int(tu[x]), int(ti[x]))
        assert np.array_equal(gi.astype(np.int64), wi) and bits_equal(gs, ws), x
        neg0 += int(((ws == 0) & np.signbit(ws)).sum())
    assert neg0 > 100
    assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti, n_threads=8))
    est.Close()
