"""Ratings added to cyclic row shards (rs_knn_update_sharded_device, ShardedKNN.Update) against a Fit of the union on
one full handle, bit for bit: every shard's rows, means and stddevs, the summed sharded predictions, and the united
sharded recommendation lists and summed score rows; growth that moves ids onto other shards and gives an empty shard
its first rows; successive updates; fold-in before the update against recommendation after it; every refusal, which
must leave every shard as it was."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import bits_equal, split
import test_recommend_gpu as trg
import test_recommend_shard_gpu as trs
from test_update_gpu import _half_stars, _new_ids

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

RS_ERR_INVALID, RS_ERR_UNSUPPORTED, RS_ERR_DUPLICATE = -1, -3, -5


def _rs():
    import recommend_sys_b200 as rs

    return rs


def _delta(est, au, ai, ar):
    """The added ratings as inner ids on the left / right sides, the extended TrainSet and its counts."""
    data = est.Data.Extend(_rs().NewRawSet(au, ai, ar))
    n0 = est.Data.Length()
    iu, ii = data.innerUsers[n0:], data.innerItems[n0:]
    if est._userBased:
        return iu, ii, data.Ratings[n0:], data.UserCount, data.ItemCount, data
    return ii, iu, data.Ratings[n0:], data.ItemCount, data.UserCount, data


def _raw_sharded(h, left, right, rating, n_left, n_right, global_mean=3.5):
    import torch

    L = _rs().core.knn_lib()
    dl = torch.tensor(np.asarray(left, dtype=np.int32), device="cuda")
    dr = torch.tensor(np.asarray(right, dtype=np.int32), device="cuda")
    dv = torch.tensor(np.asarray(rating, dtype=np.float64), device="cuda")
    torch.cuda.synchronize()
    rc = L.rs_knn_update_sharded_device(h.h, dl.data_ptr(), dr.data_ptr(), dv.data_ptr(), len(dv), n_left, n_right,
                                        global_mean)
    h.synchronize()
    return rc


def _update(shards, au, ai, ar, global_mean=None):
    """Every shard gets the same ratings, as ShardedKNN.Update gives them (GlobalMean: the extended TrainSet's unless
    given)."""
    import torch

    left, right, rating, n_left, n_right, data = _delta(shards[0], au, ai, ar)
    gm = data.GlobalMean if global_mean is None else global_mean
    dl = torch.tensor(np.asarray(left, dtype=np.int32), device="cuda")
    dr = torch.tensor(np.asarray(right, dtype=np.int32), device="cuda")
    dv = torch.tensor(np.asarray(rating, dtype=np.float64), device="cuda")
    torch.cuda.synchronize()
    for s in shards:
        s._h.update_sharded_device(dl.data_ptr(), dr.data_ptr(), dv.data_ptr(), len(dv), n_left, n_right, gm)
        s.Data, s.GlobalMean = data, gm
        s._after_fit()
    for s in shards:
        s._h.synchronize()


def _shard_rows(s):
    """The rows a shard stores, block by block in storage order (empty for a shard without rows)."""
    rows = s._h.owned_rows()
    if rows.size == 0:
        return rows, np.zeros((0, s._h.n_left))
    return rows, s.Sims


def _sharded_predict(shards, tu, ti):
    """predict_batch_sharded_device on every shard, the bit patterns summed as int64."""
    import torch

    d = shards[0].Data
    users, items = d.convert_users(tu), d.convert_items(ti)
    left, right = (users, items) if shards[0]._userBased else (items, users)
    dl = torch.tensor(np.asarray(left, dtype=np.int32), device="cuda")
    dr = torch.tensor(np.asarray(right, dtype=np.int32), device="cuda")
    acc = np.zeros(len(tu), dtype=np.uint64)
    for s in shards:
        out = torch.full((len(tu),), 7.0, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        s._h.predict_batch_sharded_device(dl.data_ptr(), dr.data_ptr(), len(tu), out.data_ptr())
        s._h.synchronize()
        acc += out.cpu().numpy().view(np.uint64)
    return acc.view(np.float64)


def _same_shards(shards, full, test=None, n_tops=(1, 10, 100)):
    """Every shard against the full handle of the union, bit for bit."""
    want = full.Sims
    for s in shards:
        assert s._h.n_left == full._h.n_left and s._h.n_right == full._h.n_right
        assert np.float64(s.GlobalMean).view(np.uint64) == np.float64(full.GlobalMean).view(np.uint64)
        rows, got = _shard_rows(s)
        assert bits_equal(got, want[rows]), s._h.params.shard_index
        if full.Means is not None:
            assert bits_equal(s.Means, full.Means)
        if full.StdDevs is not None:
            assert bits_equal(s.StdDevs, full.StdDevs)
    if test is not None:
        tu, ti, _ = split(test)
        assert bits_equal(_sharded_predict(shards, tu, ti), full.PredictBatch(tu, ti))
    side = "left" if full._userBased else "right"
    trs._check(shards, full, side, np.arange(full.Data.UserCount), n_tops)


def _close(*ests):
    for e in ests:
        e.Close()


def _configs():
    out = []
    n = 0
    for sim in ("cosine", "msd", "pearson"):
        for knn_type in ("basic", "centered", "zscore"):
            for user_based in (True, False):
                for half in (False, True):
                    out.append((sim, knn_type, user_based, half, 2 + n % 2))
                    n += 1
    return out


# ---- the tail of u1_base added to R shards of a Fit of the rest equals a Fit of all of it ----
@pytest.mark.parametrize("sim,knn_type,user_based,half,count", _configs())
def test_sharded_update_equals_refit(ml100k, sim, knn_type, user_based, half, count):
    base = ml100k["u1_base"]
    u, i, r = _half_stars(base) if half else split(base)
    m = len(r) - len(r) // 10
    extra = {"simPath": "stream"}
    shards = trs._shards(u[:m], i[:m], r[:m], sim, knn_type, user_based, "cyclic", count, extra=extra)
    _update(shards, u[m:], i[m:], r[m:])
    full = trg._fit(u, i, r, sim, knn_type, user_based, extra=extra)
    _same_shards(shards, full, ml100k["u1_test"])
    _close(full, *shards)


# ---- several updates in a row, down to single ratings ----
@pytest.mark.parametrize("sim,knn_type,user_based,count", [("pearson", "centered", True, 2), ("msd", "zscore", False, 3),
                                                           ("cosine", "basic", True, 3)])
def test_successive_sharded_updates(ml100k, sim, knn_type, user_based, count):
    base = ml100k["u1_base"]
    perm = np.random.RandomState(7).permutation(len(base))
    u, i, r = _half_stars(base[perm])
    m = len(r) - 4000
    steps = [m, m + 1, m + 2, m + 50, m + 51, m + 1000, len(r)]
    shards = trs._shards(u[:m], i[:m], r[:m], sim, knn_type, user_based, "cyclic", count)
    for a, b in zip(steps[:-1], steps[1:]):
        _update(shards, u[a:b], i[a:b], r[a:b])
    full = trg._fit(u, i, r, sim, knn_type, user_based)
    _same_shards(shards, full, ml100k["u1_test"], n_tops=(10,))
    _close(full, *shards)


# ---- growth: new ids land on the shard the block rule names ----
@pytest.mark.parametrize("user_based,new_users,new_items,count", [
    (True, [5001, 5002], [9001], 2),                     # 943 -> 945 users: past the 944 of ld_s, a new layout
    (True, list(range(5001, 5028)), [9001], 2),          # 943 -> 970 users: block 30 (ids 960..) starts on shard 0
    (True, list(range(5001, 5028)), [], 3),
    (False, [5001], [9001, 9002], 2),                    # 1682 -> 1684 items: inside the 1696 of ld_s
    (False, [5001], [9001, 9002], 3),
])
@pytest.mark.parametrize("sim,knn_type", [("pearson", "zscore"), ("msd", "centered")])
def test_sharded_growth(ml100k, user_based, new_users, new_items, count, sim, knn_type):
    base = ml100k["u1_base"]
    u, i, r = split(base)
    shards = trs._shards(u, i, r, sim, knn_type, user_based, "cyclic", count)
    n_left0 = shards[0]._h.n_left
    add = _new_ids(base, new_users, new_items, 3)
    au, ai, ar = split(add)
    _update(shards, au, ai, ar)
    assert shards[0]._h.n_left == n_left0 + (len(new_users) if user_based else len(new_items))
    full = trg._fit(np.concatenate([u, au]), np.concatenate([i, ai]), np.concatenate([r, ar]), sim, knn_type,
                    user_based)
    _same_shards(shards, full, ml100k["u1_test"], n_tops=(10,))
    # one more id on the same side: the matrix grows in place when ld_s keeps its value
    more = np.array([(7001, 50, 3), (7001, 181, 5), (1, 9101, 2), (2, 9101, 4)], dtype=np.int64)
    mu, mi, mr = split(more)
    _update(shards, mu, mi, mr)
    full2 = trg._fit(np.concatenate([u, au, mu]), np.concatenate([i, ai, mi]), np.concatenate([r, ar, mr]), sim,
                     knn_type, user_based)
    _same_shards(shards, full2, ml100k["u1_test"], n_tops=(10,))
    _close(full, full2, *shards)


def _small(n_users, n_items, per_user, seed, first_user=0):
    rng = np.random.RandomState(seed)
    rows = []
    for us in range(first_user, first_user + n_users):
        for it in rng.choice(n_items, per_user, replace=False):
            rows.append((us, it, rng.randint(1, 6)))
    return np.array(rows, dtype=np.int64)


@pytest.mark.parametrize("sim,knn_type", [("msd", "basic"), ("pearson", "zscore"), ("cosine", "centered")])
def test_empty_shard_gains_rows(sim, knn_type):
    """50 users on 3 shards: blocks 0 and 1 on shards 0 and 1, shard 2 empty.  New users 50 .. 139 fill blocks 1 .. 4,
    so shard 2 gets its first rows (block 2, ids 64 .. 95) from the update."""
    base = _small(50, 120, 12, 5)
    u, i, r = split(base)
    shards = trs._shards(u, i, r, sim, knn_type, True, "cyclic", 3, extra={"simPath": "stream"})
    assert shards[2]._h.owned_rows().size == 0
    add = _small(90, 120, 10, 6, first_user=50)
    add = np.concatenate([add, [(3, 500, 4), (64, 501, 2), (100, 500, 5)]])   # and two new items
    au, ai, ar = split(add)
    _update(shards, au, ai, ar)
    assert shards[2]._h.owned_rows().size == 32
    full = trg._fit(np.concatenate([u, au]), np.concatenate([i, ai]), np.concatenate([r, ar]), sim, knn_type, True,
                    extra={"simPath": "stream"})
    _same_shards(shards, full, n_tops=(1, 10))
    _close(full, *shards)


# ---- the touched rows in several batches ----
def test_sharded_forced_batches(ml100k, monkeypatch):
    base = ml100k["u1_base"]
    perm = np.random.RandomState(11).permutation(len(base))
    u, i, r = split(base[perm])
    m = len(r) - 2000
    for user_based in (True, False):
        shards = trs._shards(u[:m], i[:m], r[:m], "pearson", "centered", user_based, "cyclic", 3)
        monkeypatch.setenv("RS_KNN_REC_BATCH", "7")
        _update(shards, u[m:], i[m:], r[m:])
        monkeypatch.delenv("RS_KNN_REC_BATCH")
        full = trg._fit(u, i, r, "pearson", "centered", user_based)
        _same_shards(shards, full, n_tops=(10,))
        _close(full, *shards)


# ---- fold-in on a full handle before the update = sharded recommendation of the new user after it ----
@pytest.mark.parametrize("sim,knn_type", [("msd", "basic"), ("pearson", "centered"), ("cosine", "zscore")])
def test_fold_in_agrees_with_sharded_update(ml100k, sim, knn_type):
    u, i, r = split(ml100k["u1_base"])
    full = trg._fit(u, i, r, sim, knn_type, True)
    shards = trs._shards(u, i, r, sim, knn_type, True, "cyclic", 2)
    test = ml100k["u1_test"]
    rows = test[test[:, 0] == 1][:, 1:3]
    ids = full.Data.convert_items(rows[:, 0])
    raw, vals = rows[ids >= 0, 0], rows[ids >= 0, 1].astype(np.float64)
    ids = ids[ids >= 0]
    ptr = np.array([0, len(ids)], dtype=np.int64)
    want_rows = full._h.score_all_given("left", ptr, ids, vals)
    want_ids, want_top = full._h.recommend_given("left", ptr, ids, vals, 50)
    n_left = full._h.n_left
    # a new user, inner id n_left; GlobalMean stays the fitted one, as fold-in scores with it
    _update(shards, np.full(len(ids), 10 ** 6), raw, vals, full.GlobalMean)
    assert shards[0]._h.n_left == n_left + 1
    q = np.array([n_left])
    got_rows, lists, _ = trs._assemble(shards, "left", q, (50,))
    assert bits_equal(got_rows, want_rows)
    got_ids, got_top = lists[50]
    assert np.array_equal(got_ids, want_ids)
    assert bits_equal(got_top, want_top)
    _close(full, *shards)


# ---- refusals: the code, and every shard exactly as it was ----
def _snapshot(shards, test):
    tu, ti, _ = split(test)
    out = {"pred": _sharded_predict(shards, tu, ti), "n": [(s._h.n_left, s._h.n_right) for s in shards]}
    for s in shards:
        q = s._h.params.shard_index
        out[("sims", q)] = _shard_rows(s)[1]
        out[("means", q)] = s._h.means()
        if s._h.params.knn_type == _rs().core.RS_KNN_TYPE["zscore"]:
            out[("std", q)] = s._h.stddevs()
    return out


def _same_snapshot(a, b):
    assert a["n"] == b["n"]
    for key in a:
        if key != "n":
            assert bits_equal(a[key], b[key]), key


def test_sharded_refusals_leave_every_shard(ml100k):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    test = ml100k["u1_test"]
    L = rs.core.knn_lib()
    # before rs_knn_mirror
    raw = [trg._fit(u, i, r, "pearson", "zscore", True, extra={"shardCount": 2, "shardIndex": s}) for s in range(2)]
    for s in raw:
        s._h.synchronize()
        assert _raw_sharded(s._h, [0], [5], [4.0], s._h.n_left, s._h.n_right) == RS_ERR_INVALID
    _close(*raw)

    shards = trs._shards(u, i, r, "pearson", "zscore", True, "cyclic", 2)
    d = shards[0].Data
    nl, nr = shards[0]._h.n_left, shards[0]._h.n_right
    l0, r0 = int(d.innerUsers[0]), int(d.innerItems[0])            # a pair the model holds
    tl = d.convert_users(test[:3, 0])
    ti = d.convert_items(test[:3, 1])                              # pairs the model does not hold
    before = _snapshot(shards, test)
    cases = [
        (RS_ERR_INVALID, [nl], [ti[0]], [4.0], nl, nr),                  # left id out of range
        (RS_ERR_INVALID, [tl[0]], [-1], [4.0], nl, nr),                  # right id out of range
        (RS_ERR_INVALID, [tl[0]], [ti[0]], [4.0], nl - 1, nr),           # a count below the fitted one
        (RS_ERR_UNSUPPORTED, [tl[0], tl[1]], [ti[0], ti[1]], [4.0, np.nan], nl, nr),
        (RS_ERR_UNSUPPORTED, [tl[0]], [ti[0]], [3.5], nl, nr),           # not an integer: the model is RS_CLASS_INT8
        (RS_ERR_DUPLICATE, [tl[0], l0], [ti[0], r0], [4.0, 2.0], nl, nr),
        (RS_ERR_DUPLICATE, [tl[0], tl[0]], [ti[0], ti[0]], [4.0, 2.0], nl + 1, nr),
    ]
    for code, left, right, rating, n_left, n_right in cases:
        for s in shards:
            assert _raw_sharded(s._h, left, right, rating, n_left, n_right) == code, (code, left, right, rating)
        _same_snapshot(before, _snapshot(shards, test))
    # the plain entry points keep refusing cyclic shards
    for s in shards:
        left = np.array([tl[0]], np.int32)
        right = np.array([ti[0]], np.int32)
        rating = np.array([4.0])
        assert L.rs_knn_update(s._h.h, left.ctypes.data, right.ctypes.data, rating.ctypes.data, 1, nl, nr,
                               3.5) == RS_ERR_UNSUPPORTED
    _same_snapshot(before, _snapshot(shards, test))
    # and the shards still update; afterwards rs_knn_mirror is refused, and the model stays the union's
    au, ai = test[:3, 0], test[:3, 1]
    _update(shards, au, ai, np.array([4.0, 2.0, 5.0]))
    for s in shards:
        with pytest.raises(rs.core.RsError) as e:
            s._h.mirror()
        assert e.value.code == RS_ERR_INVALID
    full = trg._fit(np.concatenate([u, au]), np.concatenate([i, ai]), np.concatenate([r, [4.0, 2.0, 5.0]]),
                    "pearson", "zscore", True)
    _same_shards(shards, full, test, n_tops=(10,))

    # a full handle, and a contiguous row shard
    assert _raw_sharded(full._h, [tl[0]], [ti[0]], [4.0], nl, nr) == RS_ERR_INVALID
    contiguous = trg._fit(u, i, r, "msd", "basic", True, extra={"rowBegin": 0, "rowEnd": 500})
    snap = contiguous._h.sims_rows(0, 500)
    assert _raw_sharded(contiguous._h, [tl[0]], [ti[0]], [4.0], nl, nr) == RS_ERR_UNSUPPORTED
    assert bits_equal(contiguous._h.sims_rows(0, 500), snap)
    _close(full, contiguous, *shards)


# ---- ShardedKNN.Update over NCCL, two GPUs ----
def _nccl_worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch
    import torch.distributed as dist

    import recommend_sys_b200 as rs
    from conftest import load_ml100k

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    u, i, r = split(load_ml100k()["u1_base"])
    m = len(r) - 3000
    au = np.concatenate([u[m:], [5001, 5001]])
    ai = np.concatenate([i[m:], [1, 9001]])
    ar = np.concatenate([r[m:], [4.0, 2.0]])
    users = np.concatenate([np.unique(u)[::5], [5001, 10 ** 9]])
    for user_based in (True, False):
        params = {"sim": rs.Pearson, "userBased": user_based, "k": 40}
        est = rs.shard.ShardedKNN(rs.NewKNNWithMean(rs.Parameters(params)))
        est.Fit(rs.NewTrainSet(rs.NewRawSet(u[:m], i[:m], r[:m])))
        est.Update(rs.NewRawSet(au, ai, ar))
        with pytest.raises(rs.core.RsError):               # a pair the model holds: refused on both ranks
            est.Update(rs.NewRawSet(au[:1], ai[:1], ar[:1]))
        items, scores = est.Recommend(users, 25)
        rows = est.ScoreAll(users)
        preds = est.PredictBatch(u[:500], i[:500])
        if rank == 0:
            one = rs.NewKNNWithMean(rs.Parameters(params))
            one.Fit(rs.NewTrainSet(rs.NewRawSet(np.concatenate([u[:m], au]), np.concatenate([i[:m], ai]),
                                                np.concatenate([r[:m], ar]))))
            wi, ws = one.Recommend(users, 25)
            assert np.array_equal(items, wi) and bits_equal(scores, ws), user_based
            assert bits_equal(rows, one.ScoreAll(users)), user_based
            assert bits_equal(preds, one.PredictBatch(u[:500], i[:500])), user_based
            one.Close()
        est.Close()
    if rank == 0:
        (Path(out_dir) / "ok").write_text("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_knn_update_two_gpus(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    mp.spawn(_nccl_worker, args=(2, trs._free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok").read_text() == "ok"
