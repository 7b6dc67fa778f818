"""Recommendation for queries given as rating lists (rs_knn_score_all_given / rs_knn_recommend_given) on the device,
bit for bit: against rs_knn_score_all / rs_knn_recommend on the same handle when a list is a fitted user's own
ratings, and against the host restatement (tests/recommend_given_ref.py) for ratings the model never saw."""
import numpy as np
import pytest

from conftest import split
from recommend_given_ref import Model, lists_of_raw, user_lists
from recommend_ref import rank_rows, same_bits
import test_recommend_gpu as rg
import test_selection_gpu as sel

pytestmark = pytest.mark.gpu

RIGHT_CONFIGS = [(s, t) for s in ("cosine", "msd", "pearson", "pearson_baseline")
                 for t in ("basic", "centered", "zscore", "baseline")]
LEFT_CONFIGS = [(s, t) for s in ("cosine", "msd", "pearson") for t in ("basic", "centered", "zscore")]


def _check_lists(h, side, ptr, ids, vals, want_rows, n_tops=(1, 10, 512)):
    got = h.score_all_given(side, ptr, ids, vals)
    assert same_bits(got, want_rows)
    for n_top in n_tops:
        gi, gt = h.recommend_given(side, ptr, ids, vals, n_top)
        wi, wt = rank_rows(want_rows, n_top)
        assert np.array_equal(gi, wi), (side, n_top)
        assert same_bits(gt, wt)
    return got


def _shuffled(ptr, ids, vals, seed):
    rng = np.random.RandomState(seed)
    ids, vals = ids.copy(), vals.copy()
    for b in range(len(ptr) - 1):
        p = ptr[b] + rng.permutation(ptr[b + 1] - ptr[b])
        ids[ptr[b]:ptr[b + 1]], vals[ptr[b]:ptr[b + 1]] = ids[p], vals[p]
    return ids, vals


# ---- identity: a list equal to a fitted user's own ratings is that user's query ----
@pytest.mark.parametrize("sim,knn_type", RIGHT_CONFIGS)
def test_identity_right(ml100k, sim, knn_type):
    u, i, r = split(ml100k["u1_base"])
    extra = {"simPath": "stream"}
    if sim == "pearson_baseline":
        extra["shrinkage"] = 100.0
    est = rg._fit(u, i, r, sim, knn_type, False, extra=extra)
    h = est._h
    users, ptr, ids, vals = user_lists(u, i, r)
    want = h.score_all("right", users)
    _check_lists(h, "right", ptr, ids, vals, want)
    sids, svals = _shuffled(ptr, ids, vals, 3)                 # the order of a right list does not matter
    assert same_bits(h.score_all_given("right", ptr, sids, svals), want)
    est.Close()


@pytest.mark.parametrize("sim,knn_type", LEFT_CONFIGS)
def test_identity_left(ml100k, sim, knn_type):
    u, i, r = split(ml100k["u1_base"])
    est = rg._fit(u, i, r, sim, knn_type, True, extra={"simPath": "stream"})
    h = est._h
    users, ptr, ids, vals = user_lists(u, i, r)               # dataset order: the order Fit summed the means in
    _check_lists(h, "left", ptr, ids, vals, h.score_all("left", users))
    # the Python mirror: the train set itself, grouped by raw user, is every user in inner order
    rs = rg._rs()
    got_users, rows = est.ScoreAllGiven(rs.NewRawSet(u, i, r))
    assert np.array_equal(est.Data.convert_users(got_users), users)
    assert same_bits(rows, h.score_all("left", users))
    est.Close()


# ---- held-out ratings: lists the model never saw, against the restatement ----
HELD_OUT = [(True, "msd", "basic"), (True, "pearson", "centered"), (True, "cosine", "zscore"),
            (False, "pearson", "centered"), (False, "msd", "baseline"), (False, "cosine", "zscore")]


@pytest.mark.parametrize("user_based,sim,knn_type", HELD_OUT)
def test_held_out(ml100k, user_based, sim, knn_type):
    u, i, r = split(ml100k["u1_base"])
    tu, ti, tr = split(ml100k["u1_test"])
    est = rg._fit(u, i, r, sim, knn_type, user_based, extra={"simPath": "stream"})
    h = est._h
    side = "left" if user_based else "right"
    m = Model(u, i, r, sim, knn_type, user_based)
    ptr, ids, vals = lists_of_raw(u, i, tu, ti, tr)
    take = np.arange(0, len(ptr) - 1, 9)                     # ~100 of the users (the restatement is host Python)
    rng = np.random.RandomState(11)
    lists = []
    for b in take.tolist():
        a, e = ptr[b], ptr[b + 1]
        lists.append((ids[a:e], vals[a:e]))
        if e - a >= 1:
            lists.append((ids[a:a + 1], vals[a:a + 1]))    # a single entry
        if e - a >= 4:
            p = np.sort(rng.choice(e - a, (e - a) // 2, replace=False))
            lists.append((ids[a:e][p], vals[a:e][p]))      # a random subset
    gptr = np.concatenate([[0], np.cumsum([len(x[0]) for x in lists])]).astype(np.int64)
    gids = np.concatenate([x[0] for x in lists])
    gvals = np.concatenate([x[1] for x in lists])
    want = m.score_all_given(side, gptr, gids, gvals)
    _check_lists(h, side, gptr, gids, gvals, want, n_tops=(10, 512))
    est.Close()


# ---- hard cases ----
def test_right_list_longer_than_every_fitted_row(ml100k):
    u, i, r = split(ml100k["u1_base"])
    est = rg._fit(u, i, r, "pearson", "centered", False, extra={"simPath": "stream"})
    h = est._h
    m = Model(u, i, r, "pearson", "centered", False)
    n_items = h.n_left
    rng = np.random.RandomState(5)
    ids = np.concatenate([np.arange(n_items), rng.permutation(n_items)[:n_items - 3]])   # every item, then all but 3
    vals = rng.randint(1, 6, len(ids)).astype(np.float64)
    ptr = np.array([0, n_items, len(ids)], dtype=np.int64)
    assert n_items > np.bincount(rg._rs().NewTrainSet(rg._rs().NewRawSet(u, i, r)).innerUsers).max()
    want = m.score_all_given("right", ptr, ids, vals)
    assert np.isnan(want[0]).all() and (~np.isnan(want[1])).sum() == 3
    _check_lists(h, "right", ptr, ids, vals, want)
    ids, top = h.recommend_given("right", ptr, ids, vals, 5)
    assert (ids[0] == -1).all() and np.isnan(top[0]).all()   # a list covering every target: an empty list of results
    est.Close()


def test_left_list_without_co_raters_and_empty_lists(ml100k):
    u, i, r = split(ml100k["u1_base"])
    # items 5000 and 5001 are rated by user 9999 only: a list of them has no co-rating with any fitted user
    u2 = np.concatenate([u, [9999, 9999]])
    i2 = np.concatenate([i, [5000, 5001]])
    r2 = np.concatenate([r, [4.0, 2.0]])
    est = rg._fit(u2, i2, r2, "msd", "centered", True, extra={"simPath": "stream"})
    h = est._h
    gm = est.GlobalMean
    conv = est.Data.convert_items(np.array([5000, 5001]))
    ptr = np.array([0, 2, 2], dtype=np.int64)
    got = h.score_all_given("left", ptr, conv, np.array([5.0, 1.0]))
    assert np.isnan(got[0, conv]).all()
    rest = np.setdiff1d(np.arange(h.n_right), conv)
    assert (got[0, rest] == gm).all()                         # an all-NaN S* row: GlobalMean
    assert same_bits(got[1], h.score_all("left", [-1])[0])    # an empty list: a -1 query
    for side in ("left", "right"):
        e = rg._fit(u, i, r, "pearson", "basic", side == "left", extra={"simPath": "stream"})
        z = np.zeros(3, dtype=np.int64)
        assert same_bits(e._h.score_all_given(side, z, np.empty(0, np.int32), np.empty(0)),
                         e._h.score_all(side, [-1, -1]))
        gi, gt = e._h.recommend_given(side, z, np.empty(0, np.int32), np.empty(0), 7)
        wi, wt = e._h.recommend(side, [-1, -1], 7)
        assert np.array_equal(gi, wi) and same_bits(gt, wt)
        e.Close()
    est.Close()


def test_continuous_ratings(ml100k):
    u, i, r = split(ml100k["u1_base"])
    rng = np.random.RandomState(2)
    rc = r + rng.uniform(-0.5, 0.5, len(r)).round(3)
    tu, ti, tr = split(ml100k["u1_test"])
    trc = tr + rng.uniform(-0.5, 0.5, len(tr)).round(3)
    for user_based, sim, typ in ((True, "pearson", "zscore"), (False, "cosine", "centered")):
        est = rg._fit(u, i, rc, sim, typ, user_based, extra={"simPath": "stream"})
        side = "left" if user_based else "right"
        users, ptr, ids, vals = user_lists(u, i, rc, np.arange(0, 943, 17))
        _check_lists(est._h, side, ptr, ids, vals, est._h.score_all(side, users), n_tops=(10,))
        m = Model(u, i, rc, sim, typ, user_based)
        ptr, ids, vals = lists_of_raw(u, i, tu, ti, trc)
        sub = np.arange(0, len(ptr) - 1, 23)
        p2 = np.concatenate([[0], np.cumsum(ptr[sub + 1] - ptr[sub])]).astype(np.int64)
        ids2 = np.concatenate([ids[ptr[b]:ptr[b + 1]] for b in sub])
        vals2 = np.concatenate([vals[ptr[b]:ptr[b + 1]] for b in sub])
        _check_lists(est._h, side, p2, ids2, vals2, m.score_all_given(side, p2, ids2, vals2), n_tops=(10,))
        est.Close()


def test_signed_fixture():
    u, i, r = rg._signed_fixture()
    for user_based in (True, False):
        est = rg._fit(u, i, r, "cosine", "basic", user_based, k=2, extra={"simPath": "stream"})
        side = "left" if user_based else "right"
        users, ptr, ids, vals = user_lists(u, i, r)
        want = est._h.score_all(side, users)
        fin = want[~np.isnan(want)]
        assert np.isposinf(fin).any() and np.isneginf(fin).any()
        _check_lists(est._h, side, ptr, ids, vals, want, n_tops=(1, 5, 512))
        est.Close()


def test_selection_fixture():
    for kind in ("msd", "cosine"):
        u, i, r, left, items = sel.make_fixture(kind)
        sim = "msd" if kind == "msd" else "cosine"
        ub = rg._fit(u, i, r, sim, "centered", True, mink=sel.MINK, extra={"simPath": "stream"})
        ib = rg._fit(i, u, r, sim, "centered", False, mink=sel.MINK, extra={"simPath": "stream"})
        lq = ub.Data.convert_users(left)
        rq = ib.Data.convert_users(items)
        for k in (1, 45, 105, 256):
            for est, side, q, (uu, ii) in ((ub, "left", lq, (u, i)), (ib, "right", rq, (i, u))):
                est._h.set_k(k, sel.MINK)
                _, ptr, ids, vals = user_lists(uu, ii, r, q)
                _check_lists(est._h, side, ptr, ids, vals, est._h.score_all(side, q), n_tops=(10,))
        ub.Close()
        ib.Close()


@pytest.mark.parametrize("sim", ["cosine", "msd"])
def test_tensor_path_left(ml100k, sim):
    u, i, r = split(ml100k["u1_base"])
    est = rg._fit(u, i, r, sim, "centered", True, extra={"simPath": "tensor"})
    users, ptr, ids, vals = user_lists(u, i, r)
    _check_lists(est._h, "left", ptr, ids, vals, est._h.score_all("left", users), n_tops=(10,))
    est.Close()


def test_small_batches_and_device_variants(ml100k, monkeypatch):
    import torch

    u, i, r = split(ml100k["u1_base"])
    for user_based in (True, False):
        est = rg._fit(u, i, r, "pearson", "centered", user_based, extra={"simPath": "stream"})
        h = est._h
        side = "left" if user_based else "right"
        users, ptr, ids, vals = user_lists(u, i, r, np.arange(0, 943, 5))
        want_rows = h.score_all_given(side, ptr, ids, vals)
        want_i, want_t = h.recommend_given(side, ptr, ids, vals, 20)
        monkeypatch.setenv("RS_KNN_REC_BATCH", "3")
        assert same_bits(h.score_all_given(side, ptr, ids, vals), want_rows)
        gi, gt = h.recommend_given(side, ptr, ids, vals, 20)
        assert np.array_equal(gi, want_i) and same_bits(gt, want_t)
        monkeypatch.delenv("RS_KNN_REC_BATCH")
        dev = torch.device("cuda", torch.cuda.current_device())
        off = 5                                                 # lists that do not start at entry 0
        d_ptr = torch.from_numpy(ptr + off).to(dev)
        d_ids = torch.from_numpy(np.concatenate([np.zeros(off, np.int32), ids.astype(np.int32)])).to(dev)
        d_vals = torch.from_numpy(np.concatenate([np.full(off, np.nan), vals])).to(dev)
        n = len(ptr) - 1
        d_out = torch.empty((n, want_rows.shape[1]), dtype=torch.float64, device=dev)
        h.score_all_given_device(side, d_ptr.data_ptr(), d_ids.data_ptr(), d_vals.data_ptr(), n, d_out.data_ptr())
        d_ti = torch.empty((n, 20), dtype=torch.int32, device=dev)
        d_ts = torch.empty((n, 20), dtype=torch.float64, device=dev)
        h.recommend_given_device(side, d_ptr.data_ptr(), d_ids.data_ptr(), d_vals.data_ptr(), n, 20,
                                 d_ti.data_ptr(), d_ts.data_ptr())
        h.synchronize()
        assert same_bits(d_out.cpu().numpy(), want_rows)
        assert np.array_equal(d_ti.cpu().numpy(), want_i) and same_bits(d_ts.cpu().numpy(), want_t)
        est.Close()


# ---- refusals, host and device variants ----
def _both_refuse(h, side, ptr, ids, vals, code, n_top=5, score_all=True):
    """Host and device variants refuse the lists with `code` (score_all=False: the recommend variants only, for a
    refusal of n_top)."""
    import torch

    rs = rg._rs()
    if score_all:
        with pytest.raises(rs.RsError) as e:
            h.score_all_given(side, ptr, ids, vals)
        assert f"error {code}:" in str(e.value)
    with pytest.raises(rs.RsError) as e:
        h.recommend_given(side, ptr, ids, vals, n_top)
    assert f"error {code}:" in str(e.value)
    dev = torch.device("cuda", torch.cuda.current_device())
    ptr = np.asarray(ptr, np.int64)
    ids = np.asarray(ids, np.int32) if len(ids) else np.zeros(1, np.int32)
    vals = np.asarray(vals, np.float64) if len(vals) else np.zeros(1)
    d_ptr, d_ids, d_vals = (torch.from_numpy(x).to(dev) for x in (ptr, ids, vals))
    n = len(ptr) - 1
    d_out = torch.empty((max(1, n), max(h.n_left, h.n_right)), dtype=torch.float64, device=dev)
    d_ti = torch.empty((max(1, n), 512), dtype=torch.int32, device=dev)
    d_ts = torch.empty((max(1, n), 512), dtype=torch.float64, device=dev)
    if score_all:
        with pytest.raises(rs.RsError) as e:
            h.score_all_given_device(side, d_ptr.data_ptr(), d_ids.data_ptr(), d_vals.data_ptr(), n,
                                     d_out.data_ptr())
        assert f"error {code}:" in str(e.value)
    with pytest.raises(rs.RsError) as e:
        h.recommend_given_device(side, d_ptr.data_ptr(), d_ids.data_ptr(), d_vals.data_ptr(), n, n_top,
                                 d_ti.data_ptr(), d_ts.data_ptr())
    assert f"error {code}:" in str(e.value)


def test_refusals(ml100k):
    rs = rg._rs()
    INVALID, UNSUPPORTED, DUPLICATE = -1, -3, -5
    u, i, r = split(ml100k["u1_base"])
    est = rg._fit(u, i, r, "msd", "basic", True, extra={"simPath": "stream"})
    h = est._h
    for side in ("left", "right"):
        nt = h.n_right if side == "left" else h.n_left
        _both_refuse(h, side, [0, 2], [3, nt], [1.0, 2.0], INVALID)            # an id out of range
        _both_refuse(h, side, [0, 2], [3, -1], [1.0, 2.0], INVALID)
        _both_refuse(h, side, [0, 2, 1], [3, 4], [1.0, 2.0], INVALID)          # ptr decreasing
        _both_refuse(h, side, [0, 2], [3, 4], [1.0, np.nan], INVALID)          # a NaN rating
        _both_refuse(h, side, [0, 1, 3], [3, 4, 4], [1.0, 2.0, 3.0], DUPLICATE)
        for n_top in (0, 513):
            _both_refuse(h, side, [0, 1], [3], [1.0], INVALID, n_top=n_top, score_all=False)
        # the same id in two different lists is fine
        h.score_all_given(side, [0, 1, 2], [4, 4], [1.0, 2.0])
    h.set_k(257, 1)
    _both_refuse(h, "left", [0, 1], [3], [1.0], UNSUPPORTED)
    est.Close()
    refused = [("right", "msd", "basic", {"store": "topk", "topk": 40}),
               ("right", "msd", "basic", {"rowBegin": 0, "rowEnd": 100}),
               ("left", "msd", "baseline", {}),
               ("left", "pearson_baseline", "basic", {}),
               ("left", "pearson", "basic", {"pearsonMode": "sums"})]
    for side, sim, typ, extra in refused:
        e = rg._fit(u, i, r, sim, typ, side == "left", extra=dict(extra, simPath=extra.get("simPath", "auto")))
        _both_refuse(e._h, side, [0, 1], [3], [1.0], UNSUPPORTED)
        e.Close()
    shards = [rg._fit(u, i, r, "msd", "basic", True, extra={"shardCount": 2, "shardIndex": s}) for s in range(2)]
    for s in shards:
        s._h.peer_import_local([x._h for x in shards])
    for s in shards:
        s._h.synchronize()
    for s in shards:
        s._h.mirror()
    for s in shards:
        _both_refuse(s._h, "left", [0, 1], [3], [1.0], UNSUPPORTED)
        s.Close()
    so = rs.NewSlopeOne(rs.Parameters({}))
    so.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    _both_refuse(so._h, "right", [0, 1], [3], [1.0], UNSUPPORTED)
    so.Close()
