"""Ratings added to a fitted model (rs_knn_update, KNN.Update) against a Fit of the union on ML-100K u1, bit for bit:
the matrix, means, stddevs, predictions, score rows and recommendation lists; growth of both sides; successive
updates; fold-in before the update against recommendation after it; every refusal, which must leave the model as it
was; the memory a long sequence of updates holds."""

import numpy as np
import pytest

from conftest import bits_equal, split
from test_recommend_gpu import _fit

pytestmark = pytest.mark.gpu

RS_ERR_INVALID, RS_ERR_UNSUPPORTED, RS_ERR_DUPLICATE = -1, -3, -5


def _rs():
    import recommend_sys_b200 as rs

    return rs


def _half_stars(a):
    """u1 with every third rating lowered by half a star: a rating set that is not small integers."""
    u, i, r = split(a)
    return u, i, r - 0.5 * (np.arange(len(r)) % 3 == 0)


def _updated(u, i, r, m, sim, knn_type, user_based, extra=None, steps=None):
    """An estimator fitted on the first m rows, then updated with the rest (in `steps` slices, default one)."""
    rs = _rs()
    est = _fit(u[:m], i[:m], r[:m], sim, knn_type, user_based, extra=extra)
    bounds = steps if steps is not None else [m, len(r)]
    for a, b in zip(bounds[:-1], bounds[1:]):
        est.Update(rs.NewRawSet(u[a:b], i[a:b], r[a:b]))
    return est


def _same_model(got, want, test=None, n_tops=(1, 10, 100)):
    """Everything the two estimators answer, bit for bit."""
    assert got.Data.UserCount == want.Data.UserCount and got.Data.ItemCount == want.Data.ItemCount
    assert np.array_equal(got.Data.innerUsers, want.Data.innerUsers)
    assert np.array_equal(got.Data.innerItems, want.Data.innerItems)
    assert np.float64(got.GlobalMean).view(np.uint64) == np.float64(want.GlobalMean).view(np.uint64)
    assert bits_equal(got.Sims, want.Sims)
    if want.Means is not None:
        assert bits_equal(got.Means, want.Means)
    if want.StdDevs is not None:
        assert bits_equal(got.StdDevs, want.StdDevs)
    if test is not None:
        tu, ti, _ = split(test)
        assert bits_equal(got.PredictBatch(tu, ti), want.PredictBatch(tu, ti))
    users = np.unique(want.Data.Users)
    assert bits_equal(got.ScoreAll(users), want.ScoreAll(users))
    for n in n_tops:
        gi, gs = got.Recommend(users, n)
        wi, ws = want.Recommend(users, n)
        assert np.array_equal(gi, wi), n
        assert bits_equal(gs, ws)


def _configs():
    out = []
    for sim in ("cosine", "msd", "pearson"):
        for knn_type in ("basic", "centered", "zscore"):
            for user_based in (True, False):
                for half in (False, True):
                    paths = ("stream", "tensor") if sim != "pearson" and not half else ("stream",)
                    for path in paths:
                        out.append((sim, knn_type, user_based, half, path))
    return out


# ---- the tail of u1_base added to a Fit of the rest equals a Fit of all of it ----
@pytest.mark.parametrize("sim,knn_type,user_based,half,path", _configs())
def test_update_equals_refit(ml100k, sim, knn_type, user_based, half, path):
    base = ml100k["u1_base"]
    u, i, r = _half_stars(base) if half else split(base)
    m = len(r) - len(r) // 10
    got = _updated(u, i, r, m, sim, knn_type, user_based, extra={"simPath": path})
    want = _fit(u, i, r, sim, knn_type, user_based)
    _same_model(got, want, ml100k["u1_test"])
    got.Close()
    want.Close()


# ---- several updates in a row, down to single ratings, equal one Fit of the union ----
@pytest.mark.parametrize("sim,knn_type,user_based", [("pearson", "centered", True), ("msd", "zscore", False),
                                                     ("cosine", "basic", True)])
def test_successive_updates(ml100k, sim, knn_type, user_based):
    base = ml100k["u1_base"]
    perm = np.random.RandomState(7).permutation(len(base))
    u, i, r = _half_stars(base[perm])
    m = len(r) - 4000
    steps = [m, m + 1, m + 2, m + 50, m + 51, m + 1000, len(r)]
    got = _updated(u, i, r, m, sim, knn_type, user_based, steps=steps)
    want = _fit(u, i, r, sim, knn_type, user_based)
    _same_model(got, want, ml100k["u1_test"])
    got.Close()
    want.Close()


# ---- growth: new users and items that appear only in the added ratings ----
def _new_ids(base, users, items, seed):
    """Ratings of new users (on known and new items) and of known users on new items."""
    rng = np.random.RandomState(seed)
    known_u, known_i = np.unique(base[:, 0]), np.unique(base[:, 1])
    rows = []
    for nu in users:
        for it in rng.choice(known_i, 30, replace=False):
            rows.append((nu, it, rng.randint(1, 6)))
    for ni in items:
        for us in rng.choice(known_u, 25, replace=False):
            rows.append((us, ni, rng.randint(1, 6)))
        if users:
            rows.append((users[0], ni, 4))
    return np.array(rows, dtype=np.int64)


@pytest.mark.parametrize("user_based,new_users,new_items", [
    (True, [5001, 5002], [9001]),        # 943 -> 945 users: past the 944 of ld_s, a new layout
    (False, [5001], [9001, 9002]),       # 1682 -> 1684 items: inside the 1696 of ld_s
])
@pytest.mark.parametrize("sim,knn_type", [("pearson", "zscore"), ("msd", "centered")])
def test_growth(ml100k, user_based, new_users, new_items, sim, knn_type):
    rs = _rs()
    base = ml100k["u1_base"]
    u, i, r = split(base)
    est = _fit(u, i, r, sim, knn_type, user_based)
    n_left0 = est._h.n_left
    add = _new_ids(base, new_users, new_items, 3)
    au, ai, ar = split(add)
    est.Update(rs.NewRawSet(au, ai, ar))
    assert est._h.n_left == n_left0 + (len(new_users) if user_based else len(new_items))
    want = _fit(np.concatenate([u, au]), np.concatenate([i, ai]), np.concatenate([r, ar]), sim, knn_type, user_based)
    _same_model(est, want, ml100k["u1_test"])
    # one more id on the same side: the matrix grows in place when ld_s keeps its value
    more = np.array([(7001, 50, 3), (7001, 181, 5), (1, 9101, 2), (2, 9101, 4)], dtype=np.int64)
    mu, mi, mr = split(more)
    est.Update(rs.NewRawSet(mu, mi, mr))
    want2 = _fit(np.concatenate([u, au, mu]), np.concatenate([i, ai, mi]), np.concatenate([r, ar, mr]), sim, knn_type,
                 user_based)
    _same_model(est, want2, ml100k["u1_test"])
    for e in (est, want, want2):
        e.Close()


def test_count_growth_without_ratings(ml100k):
    """Ids beyond the rated ones get the empty rows a Fit gives them; GlobalMean is the caller's."""
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "msd", "centered", True)
    h = est._h
    n_left, n_right = h.n_left, h.n_right
    h.update(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0), n_left + 3, n_right + 2, 3.25)
    ref = _rs().core._Handle(sim="msd", knn_type="centered")
    ts = est.Data
    ref.fit(ts.innerUsers, ts.innerItems, ts.Ratings, n_left + 3, n_right + 2, 3.25)
    assert bits_equal(h.sims_rows(0, n_left + 3), ref.sims_rows(0, n_left + 3))
    assert bits_equal(h.means(), ref.means())
    q = np.arange(n_left + 3)
    assert bits_equal(h.score_all("left", q), ref.score_all("left", q))
    ref.close()
    est.Close()


# ---- fold-in before the update = recommendation by id after it (DESIGN.md §5.3c) ----
@pytest.mark.parametrize("sim,knn_type", [("msd", "basic"), ("pearson", "centered"), ("cosine", "zscore")])
def test_fold_in_agrees_with_update(ml100k, sim, knn_type):
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, sim, knn_type, True)
    h = est._h
    test = ml100k["u1_test"]
    # a new user who rates what user 1 rated in u1.test (the items the model knows), in that order
    rows = test[test[:, 0] == 1][:, 1:3]
    ids = est.Data.convert_items(rows[:, 0])
    vals = rows[ids >= 0, 1].astype(np.float64)
    ids = ids[ids >= 0]
    ptr = np.array([0, len(ids)], dtype=np.int64)
    n_left = h.n_left
    want_rows = h.score_all_given("left", ptr, ids, vals)
    want_ids, want_top = h.recommend_given("left", ptr, ids, vals, 50)
    h.update(np.full(len(ids), n_left, np.int32), ids, vals, n_left + 1, h.n_right, est.GlobalMean)
    q = np.array([n_left])
    assert bits_equal(h.score_all("left", q), want_rows)
    got_ids, got_top = h.recommend("left", q, 50)
    assert np.array_equal(got_ids, want_ids)
    assert bits_equal(got_top, want_top)
    est.Close()


# ---- refusals: the code, and a model exactly as it was ----
def _snapshot(h, test):
    tl, tr, _ = split(test)
    tl = np.minimum(tl - 1, h.n_left - 1).astype(np.int32)
    tr = np.minimum(tr - 1, h.n_right - 1).astype(np.int32)
    snap = {"sims": h.sims_rows(0, h.n_left), "means": h.means(), "pred": h.predict_batch(tl, tr),
            "n": (h.n_left, h.n_right)}
    if h.params.knn_type == _rs().core.RS_KNN_TYPE["zscore"]:
        snap["std"] = h.stddevs()
    return snap


def _same_snapshot(a, b):
    assert a["n"] == b["n"]
    for key in ("sims", "means", "pred", "std"):
        if key in a:
            assert bits_equal(a[key], b[key]), key


def _raw_update(h, left, right, rating, n_left, n_right):
    L = _rs().core.knn_lib()
    left = np.ascontiguousarray(left, dtype=np.int32)
    right = np.ascontiguousarray(right, dtype=np.int32)
    rating = np.ascontiguousarray(rating, dtype=np.float64)
    return L.rs_knn_update(h.h, left.ctypes.data, right.ctypes.data, rating.ctypes.data, len(rating), n_left, n_right,
                           3.5)


def _raw_update_device(h, left, right, rating, n_left, n_right):
    import torch

    L = _rs().core.knn_lib()
    dl = torch.tensor(np.asarray(left, dtype=np.int32), device="cuda")
    dr = torch.tensor(np.asarray(right, dtype=np.int32), device="cuda")
    dv = torch.tensor(np.asarray(rating, dtype=np.float64), device="cuda")
    torch.cuda.synchronize()
    return L.rs_knn_update_device(h.h, dl.data_ptr(), dr.data_ptr(), dv.data_ptr(), len(dv), n_left, n_right, 3.5)


def _handle(u, i, r, **kw):
    rs = _rs()
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    h = rs.core._Handle(**kw)
    h.fit(ts.innerUsers, ts.innerItems, ts.Ratings, ts.UserCount, ts.ItemCount, ts.GlobalMean)
    return h, ts


@pytest.mark.parametrize("call", [_raw_update, _raw_update_device])
def test_refusals_leave_the_model(ml100k, call):
    u, i, r = split(ml100k["u1_base"])
    test = ml100k["u1_test"]
    h, ts = _handle(u, i, r, sim="pearson", knn_type="zscore")
    nl, nr = h.n_left, h.n_right
    l0, r0 = int(ts.innerUsers[0]), int(ts.innerItems[0])          # a pair the model holds
    tl = ts.convert_users(test[:3, 0])
    ti = ts.convert_items(test[:3, 1])                             # pairs the model does not hold
    before = _snapshot(h, test)
    cases = [
        (RS_ERR_INVALID, [nl], [ti[0]], [4.0], nl, nr),                  # left id out of range
        (RS_ERR_INVALID, [tl[0]], [-1], [4.0], nl, nr),                  # right id out of range
        (RS_ERR_INVALID, [tl[0]], [ti[0]], [4.0], nl - 1, nr),           # a count below the fitted one
        (RS_ERR_INVALID, [tl[0]], [ti[0]], [4.0], nl, nr - 1),
        (RS_ERR_UNSUPPORTED, [tl[0], tl[1]], [ti[0], ti[1]], [4.0, np.nan], nl, nr),
        (RS_ERR_UNSUPPORTED, [tl[0]], [ti[0]], [3.5], nl, nr),           # not an integer: the model is RS_CLASS_INT8
        (RS_ERR_DUPLICATE, [tl[0], l0], [ti[0], r0], [4.0, 2.0], nl, nr),
        (RS_ERR_DUPLICATE, [tl[0], tl[0]], [ti[0], ti[0]], [4.0, 2.0], nl + 1, nr),
    ]
    for code, left, right, rating, n_left, n_right in cases:
        assert call(h, left, right, rating, n_left, n_right) == code, (code, left, right, rating)
        _same_snapshot(before, _snapshot(h, test))
    # and the handle still updates: the refused calls left nothing behind
    assert call(h, tl[:3], ti[:3], [4.0, 2.0, 5.0], nl, nr) == 0
    h.close()


@pytest.mark.parametrize("kw,extra", [
    (dict(sim="msd", knn_type="basic", store="topk", topk=10), {}),
    (dict(sim="msd", knn_type="basic", row_begin=0, row_end=500), {}),
    (dict(sim="pearson", knn_type="centered", pearson_mode="sums"), {}),
    (dict(sim="msd", knn_type="baseline"), {"left_bias": True}),
    (dict(sim="pearson_baseline", knn_type="centered"), {"left_bias": True, "right_bias": True}),
    (dict(sim="slope_one", knn_type="basic"), {"items_left": True}),
])
def test_refused_models(ml100k, kw, extra):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    h = rs.core._Handle(**kw)
    left, right, nl, nr = ts.innerUsers, ts.innerItems, ts.UserCount, ts.ItemCount
    if extra.get("items_left"):
        left, right, nl, nr = right, left, nr, nl
    lb = np.zeros(nl) if extra.get("left_bias") else None
    rb = np.zeros(nr) if extra.get("right_bias") else None
    h.fit(left, right, ts.Ratings, nl, nr, ts.GlobalMean, lb, rb, ts.GlobalMean if rb is not None else 0.0)
    test = ml100k["u1_test"]
    matrix = kw.get("store") != "topk" and kw["sim"] != "slope_one" and "row_end" not in kw
    before = _snapshot(h, test) if matrix else None
    assert _raw_update(h, [0], [0], [4.0], nl + 1, nr) == RS_ERR_UNSUPPORTED
    if matrix:
        _same_snapshot(before, _snapshot(h, test))
    h.close()


def test_not_fitted():
    h = _rs().core._Handle(sim="msd")
    assert _raw_update(h, [0], [0], [4.0], 1, 1) == RS_ERR_INVALID
    h.close()


# ---- the int8 planes of rs_knn_cosums answer for the union after an update ----
def test_cosums_after_update(ml100k):
    u, i, r = split(ml100k["u1_base"])
    m = len(r) - 3000
    got = _updated(u, i, r, m, "cosine", "basic", False, extra={"simPath": "tensor"})
    got._h.cosums(0, 4)                       # planes built for the fitted rows ...
    got.Update(_rs().NewRawSet(np.array([1, 2]), np.array([1682, 1681]), np.array([3.0, 4.0])))
    want = _fit(np.concatenate([u, [1, 2]]), np.concatenate([i, [1682, 1681]]), np.concatenate([r, [3.0, 4.0]]),
                "cosine", "basic", False)
    rows = [0, 100, got._h.n_left - 2]
    for row in rows:                          # ... and rebuilt for the union
        assert np.array_equal(got._h.cosums(row, 2), want._h.cosums(row, 2))
    want.Close()
    # updates alternating with rs_knn_cosums rebuild the planes in one block: the free memory stays put
    import torch

    test = ml100k["u1_test"]
    add = test[np.isin(test[:, 1], i)][:40]
    free = []
    for n, (a, b, c) in enumerate(add):
        got.Update(_rs().NewRawSet(np.array([a]), np.array([b]), np.array([float(c)])))
        got._h.cosums(0, 2)
        if n in (9, len(add) - 1):
            torch.cuda.synchronize()
            free.append(torch.cuda.mem_get_info()[0])
    assert free[0] - free[1] <= 64 << 20, free
    got.Close()


# ---- a long run of single-rating updates stops allocating ----
def test_memory_of_many_updates(ml100k):
    import torch

    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "pearson", "zscore", True)
    test = ml100k["u1_test"]
    known = np.isin(test[:, 1], i)
    add = test[known][:200]
    torch.cuda.synchronize()
    free_10 = None
    for n, (a, b, c) in enumerate(add):
        est.Update(rs.NewRawSet(np.array([a]), np.array([b]), np.array([float(c)])))
        if n == 9:
            est._h.synchronize()
            free_10 = torch.cuda.mem_get_info()[0]
    est._h.synchronize()
    free_200 = torch.cuda.mem_get_info()[0]
    bound = 64 << 20
    assert free_10 - free_200 <= bound, (free_10, free_200)
    au, ai, ar = split(add)
    want = _fit(np.concatenate([u, au]), np.concatenate([i, ai]), np.concatenate([r, ar]), "pearson", "zscore", True)
    _same_model(est, want, n_tops=(10,))
    est.Close()
    want.Close()


# ---- the touched rows in several batches ----
def test_forced_batches(ml100k, monkeypatch):
    monkeypatch.setenv("RS_KNN_REC_BATCH", "7")
    base = ml100k["u1_base"]
    perm = np.random.RandomState(11).permutation(len(base))
    u, i, r = split(base[perm])
    m = len(r) - 2000
    for user_based in (True, False):
        got = _updated(u, i, r, m, "pearson", "centered", user_based)
        monkeypatch.delenv("RS_KNN_REC_BATCH")
        want = _fit(u, i, r, "pearson", "centered", user_based)
        _same_model(got, want, n_tops=(10,))
        monkeypatch.setenv("RS_KNN_REC_BATCH", "7")
        got.Close()
        want.Close()
