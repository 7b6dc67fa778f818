"""Ratings removed from or changed in a fitted model (rs_knn_remove / rs_knn_change, KNN.Remove / KNN.Change) against
a Fit of the edited inner-id ratings with the same counts, bit for bit: the matrix, means, stddevs, predictions,
neighbour lists, top-k lists, score rows and recommendation lists; ids left without ratings and given ratings again;
edits interleaved with updates; fold-in and rs_knn_cosums after an edit; every refusal, which must leave the model as
it was; the memory a long sequence of edits holds."""

import numpy as np
import pytest

from conftest import bits_equal, split
from test_recommend_gpu import _fit
from test_update_gpu import _configs, _half_stars, _same_model, _same_snapshot, _snapshot

pytestmark = pytest.mark.gpu

RS_ERR_INVALID, RS_ERR_UNSUPPORTED, RS_ERR_DUPLICATE = -1, -3, -5


def _rs():
    import recommend_sys_b200 as rs

    return rs


def _refit(est, sim, knn_type, user_based, extra=None):
    """A Fit of the estimator's TrainSet: its ratings under its own inner ids and counts."""
    rs = _rs()
    sims = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson}
    ctors = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore}
    params = {"sim": sims[sim], "userBased": user_based, "k": 40, "mink": 1}
    params.update(extra or {})
    want = ctors[knn_type](rs.Parameters(params))
    want.Fit(est.Data)
    return want


def _same(got, want, test=None, n_tops=(1, 10, 100)):
    """_same_model, and the neighbour lists of Predict and rs_knn_topk."""
    _same_model(got, want, test, n_tops)
    gi, gs = got._h.topk(10)
    wi, ws = want._h.topk(10)
    assert np.array_equal(gi, wi) and bits_equal(gs, ws)
    for left, right in ((0, 0), (5, 17), (got._h.n_left - 1, got._h.n_right - 1)):
        a, b = got._h.predict_neighbors(left, right), want._h.predict_neighbors(left, right)
        assert np.array_equal(a[0], b[0]) and bits_equal(a[1], b[1])


def _tenth(n, seed):
    return np.sort(np.random.RandomState(seed).choice(n, n // 10, replace=False))


def _changed(r, rows, half, seed):
    new = np.random.RandomState(seed).randint(1, 6, len(rows)).astype(np.float64)
    return new - 0.5 * (np.arange(len(rows)) % 2 == 0) if half else new


# ---- a seeded tenth of u1.base removed from, or changed in, a Fit of all of it equals a Fit of the result ----
@pytest.mark.parametrize("edit", ["remove", "change"])
@pytest.mark.parametrize("sim,knn_type,user_based,half,path", _configs())
def test_edit_equals_refit(ml100k, sim, knn_type, user_based, half, path, edit):
    rs = _rs()
    base = ml100k["u1_base"]
    u, i, r = _half_stars(base) if half else split(base)
    got = _fit(u, i, r, sim, knn_type, user_based, extra={"simPath": path})
    rows = _tenth(len(r), 5)
    if edit == "remove":
        got.Remove(u[rows], i[rows])
    else:
        got.Change(rs.NewRawSet(u[rows], i[rows], _changed(r, rows, half, 6)))
    want = _refit(got, sim, knn_type, user_based)
    _same(got, want, ml100k["u1_test"])
    got.Close()
    want.Close()


# ---- a base Fit with popular columns, edited on its longest rows ----
@pytest.mark.parametrize("user_based", [True, False])
def test_edit_popular_columns(ml100k, user_based, monkeypatch):
    rs = _rs()
    monkeypatch.setenv("RS_KNN_POP_MIN", "200")
    u, i, r = split(ml100k["u1_base"])
    got = _fit(u, i, r, "pearson", "centered", user_based, extra={"simPath": "stream"})
    monkeypatch.delenv("RS_KNN_POP_MIN")
    left = u if user_based else i
    ids, counts = np.unique(left, return_counts=True)
    longest = ids[np.argsort(-counts, kind="stable")[:5]]
    rows = np.flatnonzero(np.isin(left, longest))
    rng = np.random.RandomState(8)
    rem = np.sort(rng.choice(rows, len(rows) // 3, replace=False))
    got.Remove(u[rem], i[rem])
    rest = np.setdiff1d(rows, rem)
    chg = np.sort(rng.choice(rest, len(rest) // 3, replace=False))
    got.Change(rs.NewRawSet(u[chg], i[chg], _changed(r, chg, False, 9)))
    want = _refit(got, "pearson", "centered", user_based)
    _same(got, want, ml100k["u1_test"])
    got.Close()
    want.Close()


# ---- ids left without ratings keep their rows, empty, and take ratings again under the same ids ----
@pytest.mark.parametrize("user_based", [True, False])
def test_emptied_ids_and_their_return(ml100k, user_based):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    got = _fit(u, i, r, "msd", "zscore", user_based)
    user, item = u[100], i[200]
    gone = np.flatnonzero((u == user) | (i == item))
    got.Remove(u[gone], i[gone])
    assert user not in got.Data.Users and item not in got.Data.Items
    uid, iid = got.Data.ConvertUserID(user), got.Data.ConvertItemID(item)
    lid = uid if user_based else iid
    sims = got.Sims
    assert np.isnan(sims[lid]).all() and np.isnan(sims[:, lid]).all()
    want = _refit(got, "msd", "zscore", user_based)
    _same(got, want, ml100k["u1_test"])
    q_u, q_i = np.array([user, user, u[0]]), np.array([item, i[0], item])
    assert bits_equal(got.PredictBatch(q_u, q_i), want.PredictBatch(q_u, q_i))
    want.Close()
    # an update gives them ratings again, under the same inner ids
    back = gone[: len(gone) // 2]
    got.Update(rs.NewRawSet(u[back], i[back], r[back]))
    assert got.Data.ConvertUserID(user) == uid and got.Data.ConvertItemID(item) == iid
    assert got.Data.UserCount == want.Data.UserCount and got.Data.ItemCount == want.Data.ItemCount
    want = _refit(got, "msd", "zscore", user_based)
    _same(got, want, ml100k["u1_test"])
    got.Close()
    want.Close()


# ---- the row where an id first appeared removed, then an update with new ids: no renumbering ----
def test_remove_first_appearance_then_update(ml100k):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    got = _fit(u, i, r, "pearson", "centered", True)
    got.Remove(u[:1], i[:1])                    # inner user 0 and inner item 0 first appeared here
    assert got.Data.ConvertUserID(u[0]) == 0 and got.Data.ConvertItemID(i[0]) == 0
    add = rs.NewRawSet(np.array([5001, 5001, u[0], 7, 5002]), np.array([i[0], 9001, 9001, 9002, i[5]]),
                       np.array([4.0, 3.0, 2.0, 5.0, 1.0]))
    got.Update(add)
    n_users = len(np.unique(u))
    assert got.Data.ConvertUserID(5001) == n_users and got.Data.UserCount == n_users + 2
    want = _refit(got, "pearson", "centered", True)
    _same(got, want, ml100k["u1_test"])
    got.Close()
    want.Close()


# ---- update -> remove -> change -> update -> remove on a z-score model of half stars ----
@pytest.mark.parametrize("user_based", [True, False])
def test_interleaved_with_updates(ml100k, user_based):
    rs = _rs()
    base = ml100k["u1_base"]
    perm = np.random.RandomState(12).permutation(len(base))
    u, i, r = _half_stars(base[perm])
    m = len(r) - 3000
    got = _fit(u[:m], i[:m], r[:m], "cosine", "zscore", user_based)
    test = ml100k["u1_test"]
    got.Update(rs.NewRawSet(u[m:m + 2000], i[m:m + 2000], r[m:m + 2000]))
    rem = np.concatenate([np.arange(0, m, 97), np.arange(m, m + 2000, 13)])    # old pairs and added ones
    got.Remove(u[rem], i[rem])
    kept = np.setdiff1d(np.arange(m + 2000), rem)
    chg = kept[::41]
    got.Change(rs.NewRawSet(u[chg], i[chg], _changed(r, chg, True, 13)))
    got.Update(rs.NewRawSet(u[m + 2000:], i[m + 2000:], r[m + 2000:]))
    rem2 = np.concatenate([chg[::3], np.arange(m + 2000, len(r), 7)])          # changed pairs and the newest
    got.Remove(u[rem2], i[rem2])
    want = _refit(got, "cosine", "zscore", user_based)
    _same(got, want, test)
    got.Close()
    want.Close()


# ---- fold-in on the edited model equals fold-in on the refit ----
@pytest.mark.parametrize("sim,knn_type", [("msd", "basic"), ("pearson", "centered"), ("cosine", "zscore")])
def test_fold_in_after_edit(ml100k, sim, knn_type):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    got = _fit(u, i, r, sim, knn_type, True)
    rows = _tenth(len(r), 21)
    got.Remove(u[rows[::2]], i[rows[::2]])
    got.Change(rs.NewRawSet(u[rows[1::2]], i[rows[1::2]], _changed(r, rows[1::2], False, 22)))
    want = _refit(got, sim, knn_type, True)
    test = ml100k["u1_test"]
    rows_t = test[test[:, 0] == 1][:, 1:3]
    ids = got.Data.convert_items(rows_t[:, 0])
    vals = rows_t[ids >= 0, 1].astype(np.float64)
    ids = ids[ids >= 0]
    ptr = np.array([0, len(ids)], dtype=np.int64)
    for side, q_ids in (("left", ids), ("right", got.Data.convert_users(np.array([1, 2, 3])))):
        q_vals = vals if side == "left" else np.array([4.0, 2.0, 5.0])
        q_ptr = ptr if side == "left" else np.array([0, 3], dtype=np.int64)
        assert bits_equal(got._h.score_all_given(side, q_ptr, q_ids, q_vals),
                          want._h.score_all_given(side, q_ptr, q_ids, q_vals))
        gi, gs = got._h.recommend_given(side, q_ptr, q_ids, q_vals, 50)
        wi, ws = want._h.recommend_given(side, q_ptr, q_ids, q_vals, 50)
        assert np.array_equal(gi, wi) and bits_equal(gs, ws)
    got.Close()
    want.Close()


# ---- the int8 planes of rs_knn_cosums answer for the edited ratings ----
def test_cosums_after_edit(ml100k):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    got = _fit(u, i, r, "cosine", "basic", False, extra={"simPath": "tensor"})
    got._h.cosums(0, 4)
    rows = _tenth(len(r), 31)
    got.Remove(u[rows[::2]], i[rows[::2]])
    got.Change(rs.NewRawSet(u[rows[1::2]], i[rows[1::2]], _changed(r, rows[1::2], False, 32)))
    want = _refit(got, "cosine", "basic", False, extra={"simPath": "tensor"})
    for row in (0, 100, got._h.n_left - 2):
        assert np.array_equal(got._h.cosums(row, 2), want._h.cosums(row, 2))
    got.Close()
    want.Close()


# ---- the touched rows in several batches ----
def test_forced_batches(ml100k, monkeypatch):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    for user_based in (True, False):
        got = _fit(u, i, r, "pearson", "centered", user_based)
        rows = _tenth(len(r), 41)
        monkeypatch.setenv("RS_KNN_REC_BATCH", "7")
        got.Remove(u[rows[::2]], i[rows[::2]])
        got.Change(rs.NewRawSet(u[rows[1::2]], i[rows[1::2]], _changed(r, rows[1::2], False, 42)))
        monkeypatch.delenv("RS_KNN_REC_BATCH")
        want = _refit(got, "pearson", "centered", user_based)
        _same(got, want, n_tops=(10,))
        got.Close()
        want.Close()


# ---- refusals: the code, and a model exactly as it was ----
def _arrays(left, right, rating=None):
    out = [np.ascontiguousarray(left, dtype=np.int32), np.ascontiguousarray(right, dtype=np.int32)]
    if rating is not None:
        out.append(np.ascontiguousarray(rating, dtype=np.float64))
    return out


def _host(h, left, right, rating=None):
    L = _rs().core.knn_lib()
    a = _arrays(left, right, rating)
    if rating is None:
        return L.rs_knn_remove(h.h, a[0].ctypes.data, a[1].ctypes.data, len(a[0]), 3.5)
    return L.rs_knn_change(h.h, a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data, len(a[0]), 3.5)


def _device(h, left, right, rating=None):
    import torch

    L = _rs().core.knn_lib()
    d = [torch.tensor(x, device="cuda") for x in _arrays(left, right, rating)]
    torch.cuda.synchronize()
    if rating is None:
        return L.rs_knn_remove_device(h.h, d[0].data_ptr(), d[1].data_ptr(), len(d[0]), 3.5)
    return L.rs_knn_change_device(h.h, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), len(d[0]), 3.5)


def _handle(u, i, r, **kw):
    rs = _rs()
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    h = rs.core._Handle(**kw)
    h.fit(ts.innerUsers, ts.innerItems, ts.Ratings, ts.UserCount, ts.ItemCount, ts.GlobalMean)
    return h, ts


@pytest.mark.parametrize("call", [_host, _device])
def test_refusals_leave_the_model(ml100k, call):
    u, i, r = split(ml100k["u1_base"])
    test = ml100k["u1_test"]
    h, ts = _handle(u, i, r, sim="pearson", knn_type="zscore")
    nl, nr = h.n_left, h.n_right
    held_l, held_r = ts.innerUsers[:3], ts.innerItems[:3]              # pairs the model holds
    tl, ti = ts.convert_users(test[:3, 0]), ts.convert_items(test[:3, 1])
    assert not np.isin(tl.astype(np.int64) * nr + ti, ts.innerUsers.astype(np.int64) * nr + ts.innerItems).any()
    before = _snapshot(h, test)
    cases = [
        (RS_ERR_INVALID, [nl], [held_r[0]], None),                       # left id out of range
        (RS_ERR_INVALID, [held_l[0]], [-1], None),                       # right id out of range
        (RS_ERR_INVALID, [held_l[0], tl[0]], [held_r[0], ti[0]], None),  # a pair the model does not hold
        (RS_ERR_INVALID, ts.innerUsers, ts.innerItems, None),            # nothing would be left
        (RS_ERR_DUPLICATE, [held_l[0], held_l[0]], [held_r[0], held_r[0]], None),
        (RS_ERR_INVALID, [nl], [held_r[0]], [4.0]),
        (RS_ERR_INVALID, [tl[0]], [ti[0]], [4.0]),
        (RS_ERR_DUPLICATE, [held_l[1], held_l[1]], [held_r[1], held_r[1]], [4.0, 2.0]),
        (RS_ERR_UNSUPPORTED, held_l[:2], held_r[:2], [4.0, np.nan]),
        (RS_ERR_UNSUPPORTED, held_l[:1], held_r[:1], [3.5]),              # not an integer: RS_CLASS_INT8
        (RS_ERR_UNSUPPORTED, held_l[:1], held_r[:1], [12.0]),             # outside [-11, 11]
    ]
    for code, left, right, rating in cases:
        assert call(h, left, right, rating) == code, (code, left, right, rating)
        _same_snapshot(before, _snapshot(h, test))
    L = _rs().core.knn_lib()
    assert L.rs_knn_remove(h.h, None, None, 1, 3.5) == RS_ERR_INVALID     # null pointers with n > 0
    assert L.rs_knn_change(h.h, None, None, None, 1, 3.5) == RS_ERR_INVALID
    _same_snapshot(before, _snapshot(h, test))
    # and the handle still edits: the refused calls left nothing behind
    assert call(h, held_l, held_r, [4.0, 2.0, 5.0]) == 0
    assert call(h, held_l[:2], held_r[:2]) == 0
    h.close()


@pytest.mark.parametrize("kw,extra", [
    (dict(sim="msd", knn_type="basic", store="topk", topk=10), {}),
    (dict(sim="msd", knn_type="basic", row_begin=0, row_end=500), {}),
    (dict(sim="msd", knn_type="basic", shard_count=2, shard_index=0), {}),
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
    matrix = (kw.get("store") != "topk" and kw["sim"] != "slope_one" and "row_end" not in kw
              and "shard_count" not in kw)
    before = _snapshot(h, test) if matrix else None
    for call in (_host, _device):
        assert call(h, left[:2], right[:2]) == RS_ERR_UNSUPPORTED
        assert call(h, left[:2], right[:2], [4.0, 2.0]) == RS_ERR_UNSUPPORTED
        if matrix:
            _same_snapshot(before, _snapshot(h, test))
    h.close()


def test_not_fitted():
    h = _rs().core._Handle(sim="msd")
    assert _host(h, [0], [0]) == RS_ERR_INVALID
    assert _host(h, [0], [0], [4.0]) == RS_ERR_INVALID
    h.close()


def test_knn_refusal_leaves_the_estimator(ml100k):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "msd", "centered", True)
    data, gm, means = est.Data, est.GlobalMean, est.Means
    with pytest.raises(rs.core.RsError) as e:
        est.Remove([u[0], 10 ** 6], [i[0], i[1]])            # an unknown raw id: refused before any device call
    assert e.value.code == RS_ERR_INVALID
    with pytest.raises(rs.core.RsError) as e:
        est.Change(rs.NewRawSet([u[0]], [i[0]], [np.nan]))  # refused by the device
    assert e.value.code == RS_ERR_UNSUPPORTED
    assert est.Data is data and est.GlobalMean == gm and est.Means is means
    est.Close()


# ---- a long run of single-pair edits stops allocating ----
def test_memory_of_many_edits(ml100k):
    import torch

    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    est = _fit(u, i, r, "pearson", "zscore", True)
    picks = np.random.RandomState(51).choice(len(r), 200, replace=False)
    torch.cuda.synchronize()
    free_10 = None
    for n, x in enumerate(picks):
        if n % 2 == 0:
            est.Remove(u[x:x + 1], i[x:x + 1])
        else:
            est.Change(rs.NewRawSet(u[x:x + 1], i[x:x + 1], np.array([float(6 - r[x])])))
        if n == 9:
            est._h.synchronize()
            free_10 = torch.cuda.mem_get_info()[0]
    est._h.synchronize()
    free_200 = torch.cuda.mem_get_info()[0]
    assert free_10 - free_200 <= 64 << 20, (free_10, free_200)
    want = _refit(est, "pearson", "zscore", True)
    _same(est, want, n_tops=(10,))
    est.Close()
    want.Close()
