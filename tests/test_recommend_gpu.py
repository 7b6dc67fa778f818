"""Top-N recommendation on the device (rs_knn_score_all / rs_knn_recommend) against the oracle and against
rs_knn_predict_batch on the same handle, bit for bit."""
import numpy as np
import pytest

from conftest import split
from oracle import binding as ob
from recommend_ref import rank_rows, same_bits, score_all
import test_selection_gpu as sel

pytestmark = pytest.mark.gpu

SIM_NAMES = ("cosine", "msd", "pearson")
KNN_TYPES = ("basic", "centered", "zscore", "baseline")


def _rs():
    import recommend_sys_b200 as rs

    return rs


def _fit(u, i, r, sim, knn_type, user_based, k=40, mink=1, extra=None):
    rs = _rs()
    sims = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson, "pearson_baseline": rs.PearsonBaseline}
    ctors = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore,
             "baseline": rs.NewKNNBaseLine}
    params = {"sim": sims[sim], "userBased": user_based, "k": k, "mink": mink}
    params.update(extra or {})
    est = ctors[knn_type](rs.Parameters(params))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    return est


def _predict_rows(h, side, queries, n_targets):
    """score rows through rs_knn_predict_batch: every (query, target) pair, rated targets still scored."""
    q = np.repeat(np.asarray(queries, dtype=np.int32), n_targets)
    t = np.tile(np.arange(n_targets, dtype=np.int32), len(queries))
    left, right = (q, t) if side == "left" else (t, q)
    return h.predict_batch(left, right).reshape(len(queries), n_targets)


def _check_handle(h, side, queries, n_tops, want=None):
    """score_all against predict_batch (+ NaN on rated targets) and, if given, the oracle rows; recommend against
    the ranking rule on those rows."""
    got = h.score_all(side, queries)
    pred = _predict_rows(h, side, queries, got.shape[1])
    rated = np.isnan(got) & ~np.isnan(pred)
    assert same_bits(np.where(np.isnan(got), np.nan, pred), got)
    if want is not None:
        assert same_bits(got, want)
        assert np.array_equal(np.isnan(want), np.isnan(got))
    for n_top in n_tops:
        ids, top = h.recommend(side, queries, n_top)
        wi, wt = rank_rows(got, n_top)
        assert np.array_equal(ids, wi), (side, n_top)
        assert same_bits(top, wt)
    return got, rated


# ---- ML-100K u1: all users, all targets, both orientations, every sim x KNN type ----
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", SIM_NAMES)
@pytest.mark.parametrize("knn_type", KNN_TYPES)
def test_ml100k_every_user(ml100k, sim, knn_type, user_based):
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, sim, knn_type, user_based, extra={"simPath": "stream"})
    side = "left" if user_based else "right"
    n_users = est.Data.UserCount
    queries = np.arange(n_users)
    ref = ob.KNN(sim=sim, knn_type=knn_type, user_based=user_based, k=40, min_k=1, n_jobs=8,
                 tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    want = score_all(ref, u, i, user_based, side, queries)
    _check_handle(est._h, side, queries, (1, 10, 512), want)
    est.Close()


# ---- the designed selection fixture at every k ----
@pytest.mark.parametrize("kind", ["msd", "cosine"])
@pytest.mark.parametrize("knn_type", ["basic", "centered"])
def test_selection_fixture_every_k(kind, knn_type):
    u, i, r, left, items = sel.make_fixture(kind)
    sim = "msd" if kind == "msd" else "cosine"
    ub = _fit(u, i, r, sim, knn_type, True, mink=sel.MINK, extra={"simPath": "stream"})
    ib = _fit(i, u, r, sim, knn_type, False, mink=sel.MINK, extra={"simPath": "stream"})   # users <-> items
    ts = ub.Data
    lq = ts.convert_users(left)                               # the pattern rows, left queries
    rq = ib.Data.convert_users(items)                         # the test items, as the right side of the swap
    for k in sel.K_SWEEP:
        for est, side, q, ubased, (uu, ii) in ((ub, "left", lq, True, (u, i)), (ib, "right", rq, False, (i, u))):
            est._h.set_k(k, sel.MINK)
            ref = ob.KNN(sim=sim, knn_type=knn_type, user_based=ubased, k=k, min_k=sel.MINK, n_jobs=8,
                         tie_policy="canonical").fit(ob.TrainSet(uu, ii, r))
            want = score_all(ref, uu, ii, ubased, side, q)
            _check_handle(est._h, side, q, (10,), want)
    ub.Close()
    ib.Close()


# ---- non-finite and signed scores ----
def _signed_fixture():
    """Cosine on +-1 ratings with k = 2: two neighbours of similarity +1 and -1 cancel (sum of weights 0), which
    gives +Inf, -Inf and NaN scores; exact zeros, -0.0 among them, occur too."""
    rng = np.random.RandomState(7)
    u, i, r = [], [], []
    for uu in range(40):
        for ii in rng.choice(30, 8, replace=False):
            u.append(uu); i.append(int(ii)); r.append(float(rng.choice([-1.0, 1.0])))
    return np.array(u, dtype=np.int64), np.array(i, dtype=np.int64), np.array(r)


def test_non_finite_and_signed_scores():
    u, i, r = _signed_fixture()
    neg0 = 0
    for user_based in (True, False):
        est = _fit(u, i, r, "cosine", "basic", user_based, k=2, extra={"simPath": "stream"})
        side = "left" if user_based else "right"
        q = np.arange(est._h.n_left if side == "left" else est._h.n_right)
        ref = ob.KNN(sim="cosine", knn_type="basic", user_based=user_based, k=2, min_k=1, n_jobs=8,
                     tie_policy="canonical").fit(ob.TrainSet(u, i, r))
        want = score_all(ref, u, i, user_based, side, q)
        got, rated = _check_handle(est._h, side, q, (1, 5, 512), want)
        fin = got[~np.isnan(got)]
        assert np.isposinf(fin).any() and np.isneginf(fin).any() and (np.isnan(got) & ~rated).any()
        assert (fin == 0).any()
        is_neg0 = lambda x: x.view(np.uint64) == np.uint64(0x8000000000000000)
        ids, top = est._h.recommend(side, q, 512)
        # every score is listed (n_top >= targets): each -0.0 score is listed as -0.0, at its (key, id) place
        assert np.array_equal(is_neg0(got).sum(axis=1), is_neg0(top).sum(axis=1))
        neg0 += int(is_neg0(got).sum())
        assert not np.isnan(top[ids >= 0]).any()
        for b in range(len(q)):
            n = (ids[b] >= 0).sum()
            assert n == (~np.isnan(got[b])).sum()
            row = top[b, :n]
            pinf, ninf = np.isposinf(row), np.isneginf(row)
            assert not pinf.any() or pinf[:pinf.sum()].all()      # +Inf first
            assert not ninf.any() or ninf[n - ninf.sum():].all()  # -Inf last
        est.Close()
    assert neg0 > 0                                       # wrat = +0 over wsum < 0: the fixture has -0.0 scores


def test_negative_zero_scores_are_reported(ml100k):
    """PearsonBaseline with shrinkage: the similarities include exact -0.0 (the candidates' keys fold it to +0.0,
    as Predict's do).  The -0.0 scores themselves are covered by test_non_finite_and_signed_scores."""
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "pearson_baseline", "basic", False, extra={"simPath": "stream", "shrinkage": 100.0})
    q = np.arange(200)
    got, _ = _check_handle(est._h, "right", q, (512,))
    est.Close()


# ---- tensor path and Pearson sums ----
@pytest.mark.parametrize("sim,extra", [("cosine", {"simPath": "tensor"}), ("msd", {"simPath": "tensor"}),
                                       ("pearson", {"pearsonMode": "sums"})])
def test_other_paths(ml100k, sim, extra):
    u, i, r = split(ml100k["u1_base"])
    for user_based in (True, False):
        est = _fit(u, i, r, sim, "centered", user_based, extra=extra)
        side = "left" if user_based else "right"
        _check_handle(est._h, side, np.arange(300), (10, 512))
        est.Close()


# ---- edge cases ----
def test_edge_cases(ml100k, monkeypatch):
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "pearson", "centered", False, extra={"simPath": "stream"})
    h = est._h
    n_items = h.n_left
    # n = 0
    ids, top = h.recommend("right", np.empty(0, np.int32), 10)
    assert ids.shape == (0, 10)
    assert h.score_all("right", np.empty(0, np.int32)).shape == (0, n_items)
    # the -1 query: GlobalMean everywhere, the first n_top ids
    s = h.score_all("right", [-1])
    assert (s == est.GlobalMean).all()
    ids, top = h.recommend("right", [-1, -1], 7)
    assert (ids == np.arange(7)).all() and (top == est.GlobalMean).all()
    # duplicates in one call, padding beyond the unrated targets
    q = np.array([5, 5, 17, 5])
    ids, top = h.recommend("right", q, 512)
    assert np.array_equal(ids[0], ids[1]) and np.array_equal(ids[0], ids[3]) and same_bits(top[0], top[3])
    # several slab batches
    q = np.arange(0, 943, 7)
    want_ids, want_top = h.recommend("right", q, 20)
    monkeypatch.setenv("RS_KNN_REC_BATCH", "3")
    got_ids, got_top = h.recommend("right", q, 20)
    assert np.array_equal(want_ids, got_ids) and same_bits(want_top, got_top)
    monkeypatch.delenv("RS_KNN_REC_BATCH")
    est.Close()


def test_query_that_rated_every_target():
    u = np.array([0] * 6 + [1, 1, 2, 2, 3], dtype=np.int64)
    i = np.array([0, 1, 2, 3, 4, 5, 0, 1, 2, 3, 4], dtype=np.int64)
    r = np.array([1, 2, 3, 4, 5, 1, 2, 3, 4, 5, 1], dtype=np.float64)
    est = _fit(u, i, r, "msd", "basic", True, extra={"simPath": "stream"})
    ids, top = est._h.recommend("left", [0, 1], 8)
    assert (ids[0] == -1).all() and np.isnan(top[0]).all()
    assert (ids[1, 4:] == -1).all() and (ids[1, :4] >= 0).all()
    est.Close()


def test_python_mirror_maps_raw_ids(ml100k):
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "pearson", "centered", False, extra={"simPath": "stream"})
    users = np.array([1, 5, 943, 10 ** 9])                   # the last one is unknown: newID
    items, scores = est.Recommend(users, 15)
    q = est.Data.convert_users(users)
    ids, top = est._h.recommend("right", q, 15)
    raw = np.empty(est.Data.ItemCount, np.int64)
    raw[est.Data.innerItems] = est.Data.Items
    assert np.array_equal(items, np.where(ids >= 0, raw[np.maximum(ids, 0)], -1)) and same_bits(scores, top)
    full = est.ScoreAll(users)
    for b, user in enumerate(users[:3]):
        pred = est.PredictBatch(np.full(5, user), raw[ids[b, :5]])
        assert same_bits(pred, full[b, ids[b, :5]])
    est.Close()


# ---- refusals ----
def test_refusals(ml100k):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "msd", "basic", True, extra={"simPath": "stream"})
    h = est._h
    for n_top in (0, 513):
        with pytest.raises(RuntimeError):
            h.recommend("left", [0], n_top)
    for bad in (-2, h.n_left):
        with pytest.raises(RuntimeError):
            h.recommend("left", [bad], 5)
        with pytest.raises(RuntimeError):
            h.score_all("left", [bad])
    h.set_k(257, 1)
    with pytest.raises(RuntimeError):
        h.recommend("left", [0], 5)
    with pytest.raises(RuntimeError):
        h.score_all("left", [0])
    est.Close()
    for extra in ({"store": "topk", "topk": 40}, {"rowBegin": 0, "rowEnd": 100}):
        e = _fit(u, i, r, "msd", "basic", True, extra=dict(extra, simPath="stream"))
        with pytest.raises(RuntimeError):
            e._h.recommend("left", [0], 5)
        e.Close()
    # cyclic row shards, two on one GPU
    shards = [_fit(u, i, r, "msd", "basic", True, extra={"shardCount": 2, "shardIndex": s}) for s in range(2)]
    for s in shards:
        s._h.peer_import_local([x._h for x in shards])
    for s in shards:
        s._h.synchronize()
    for s in shards:
        s._h.mirror()
    for s in shards:
        with pytest.raises(RuntimeError):
            s._h.recommend("left", [0], 5)
        s.Close()
    so = rs.NewSlopeOne(rs.Parameters({}))
    so.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    with pytest.raises(RuntimeError):
        so._h.recommend("right", [0], 5)
    so.Close()
