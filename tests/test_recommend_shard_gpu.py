"""Top-N recommendation on row shards (rs_knn_score_all_sharded_device / rs_knn_recommend_sharded_device): the
shards of one matrix live on one GPU, each answers the same queries, and the assembled result — integer sum of the
score rows' bit patterns, union of the partial lists — must equal rs_knn_score_all / rs_knn_recommend of one full
handle, and the oracle, bit for bit."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import split
from oracle import binding as ob
from recommend_ref import rank_rows, same_bits, score_all
import test_recommend_gpu as trg
import test_selection_gpu as sel

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _rs():
    import recommend_sys_b200 as rs

    return rs


def _n_left(u, i, user_based):
    return len(np.unique(u if user_based else i))


def _shards(u, i, r, sim, knn_type, user_based, scheme, count, k=40, mink=1, extra=None):
    """`count` row shards of one Fit on the current GPU: cyclic (wired with peer_import_local + mirror) or contiguous
    (shard.shard_rows bounds)."""
    rs = _rs()
    extra = dict(extra or {})
    out = []
    for s in range(count):
        if scheme == "cyclic":
            e = dict(extra, shardCount=count, shardIndex=s)
        else:
            b, end = rs.shard.shard_rows(_n_left(u, i, user_based), count, s)
            e = dict(extra, rowBegin=b, rowEnd=end)
        out.append(trg._fit(u, i, r, sim, knn_type, user_based, k=k, mink=mink, extra=e))
    if scheme == "cyclic":
        for s in out:
            s._h.synchronize()
        for s in out:
            s._h.peer_import_local([x._h for x in out])
            s._h.mirror()
    return out


def _assemble(shards, side, queries, n_tops):
    """Every shard answers the same queries; (score rows summed as 64-bit integers, {n_top: united lists}, {n_top:
    partial lists [shard][query][n_top]})."""
    import torch

    from recommend_sys_b200.shard import union_recommend_device

    h0 = shards[0]._h
    n = len(queries)
    nt = h0._n_targets(_rs().core.RS_SIDE[side])
    dq = torch.from_numpy(np.ascontiguousarray(queries, dtype=np.int32)).cuda()
    torch.cuda.synchronize()
    acc = np.zeros((n, nt), dtype=np.uint64)
    for s in shards:
        out = torch.full((n, nt), 7.0, dtype=torch.float64, device="cuda")     # every cell must be written
        torch.cuda.synchronize()
        s._h.score_all_sharded_device(side, dq.data_ptr(), n, out.data_ptr())
        s._h.synchronize()
        acc += out.cpu().numpy().view(np.uint64)
    lists, parts = {}, {}
    for n_top in n_tops:
        ai = torch.full((len(shards), n, n_top), 7, dtype=torch.int32, device="cuda")
        as_ = torch.full((len(shards), n, n_top), 7.0, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        for j, s in enumerate(shards):
            s._h.recommend_sharded_device(side, dq.data_ptr(), n, n_top, ai[j].data_ptr(), as_[j].data_ptr())
            s._h.synchronize()
        ui, us = union_recommend_device(ai, as_)
        torch.cuda.synchronize()
        lists[n_top] = (ui.cpu().numpy(), us.cpu().numpy())
        parts[n_top] = (ai.cpu().numpy(), as_.cpu().numpy())
    return acc.view(np.float64), lists, parts


def _check(shards, full, side, queries, n_tops, want=None):
    """The assembled result against the full handle (queries out of range there as -1) and, if given, the oracle."""
    n_side = full._h.n_left if side == "left" else full._h.n_right
    q = np.asarray(queries)
    q_full = np.where((q >= 0) & (q < n_side), q, -1)
    rows, lists, parts = _assemble(shards, side, q, n_tops)
    full_rows = full._h.score_all(side, q_full)
    assert same_bits(rows, full_rows), side
    if want is not None:
        assert same_bits(rows, want)
    for n_top in n_tops:
        ids, top = lists[n_top]
        wi, wt = full._h.recommend(side, q_full, n_top)
        assert np.array_equal(ids, wi), (side, n_top)
        assert same_bits(top, wt)
        ri, rt = rank_rows(full_rows, n_top)
        assert np.array_equal(ids, ri) and same_bits(top, rt)
        pi, ps = parts[n_top]
        assert (pi >= -1).all() and np.isnan(ps[pi < 0]).all()          # unused slots: -1 / NaN
        if side == "left":                                # each list is produced by one shard only
            assert ((pi[:, :, 0] >= 0).sum(axis=0) <= 1).all()
    return rows, parts


def _close(*ests):
    for e in ests:
        e.Close()


# ---- ML-100K u1: both orientations, cyclic and contiguous shards, several sims / KNN types / n_top ----
CASES = [
    ("cyclic", 2, "msd", "basic", {"simPath": "stream"}, (1, 10, 512)),
    ("cyclic", 3, "pearson", "centered", {"simPath": "stream"}, (1, 10, 512)),
    ("contiguous", 2, "msd", "centered", {"simPath": "stream"}, (1, 10, 512)),
    ("contiguous", 2, "cosine", "basic", {"simPath": "tensor"}, (10, 512)),
    ("cyclic", 5, "pearson", "basic", {"simPath": "stream"}, (512,)),       # 5 x 512 > 2048: the tree union
]


@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("scheme,count,sim,knn_type,extra,n_tops", CASES)
def test_ml100k_shards(ml100k, scheme, count, sim, knn_type, extra, n_tops, user_based):
    u, i, r = split(ml100k["u1_base"])
    full = trg._fit(u, i, r, sim, knn_type, user_based, extra=extra)
    shards = _shards(u, i, r, sim, knn_type, user_based, scheme, count, extra=extra)
    side = "left" if user_based else "right"
    users = np.arange(full.Data.UserCount)
    want = None
    if extra.get("simPath") == "stream":
        ref = ob.KNN(sim=sim, knn_type=knn_type, user_based=user_based, k=40, min_k=1, n_jobs=8,
                     tie_policy="canonical").fit(ob.TrainSet(u, i, r))
        want = score_all(ref, u, i, user_based, side, users)
    _check(shards, full, side, users, n_tops, want)
    # cold start: -1 and ids out of range on both sides, mixed with known queries; each list comes out once
    q = np.array([-1, 3, -1, len(users), 700, -7, 2 ** 30])
    _check(shards, full, side, q, (5, 512))
    _close(full, *shards)


# ---- +-1 Cosine: NaN, +-Inf and -0.0 scores; item-based, shard 1 holds no rows ----
def test_signed_scores_two_shards():
    u, i, r = trg._signed_fixture()
    neg0 = 0
    for user_based in (True, False):
        full = trg._fit(u, i, r, "cosine", "basic", user_based, k=2, extra={"simPath": "stream"})
        shards = _shards(u, i, r, "cosine", "basic", user_based, "cyclic", 2, k=2, extra={"simPath": "stream"})
        side = "left" if user_based else "right"
        q = np.arange(full._h.n_left if side == "left" else full._h.n_right)
        ref = ob.KNN(sim="cosine", knn_type="basic", user_based=user_based, k=2, min_k=1, n_jobs=8,
                     tie_policy="canonical").fit(ob.TrainSet(u, i, r))
        want = score_all(ref, u, i, user_based, side, q)
        rows, parts = _check(shards, full, side, q, (1, 5, 512), want)
        neg0 += int((rows.view(np.uint64) == np.uint64(0x8000000000000000)).sum())
        if not user_based:                                # 30 items: one block of 32, all on shard 0
            assert shards[1]._h.owned_rows().size == 0
            pi, ps = parts[5]
            assert (pi[1] == -1).all() and np.isnan(ps[1]).all()
            out, _, _ = _assemble(shards[1:], side, q, ())
            assert (out.view(np.uint64) == 0).all()
        _close(full, *shards)
    assert neg0 > 0                                       # -0.0 scores survive the integer sum


# ---- the selection fixture at k = 256 ----
def test_selection_fixture_k256():
    kind, knn_type = "msd", "centered"
    u, i, r, left, items = sel.make_fixture(kind)
    for user_based, (uu, ii) in ((True, (u, i)), (False, (i, u))):
        extra = {"simPath": "stream"}
        full = trg._fit(uu, ii, r, "msd", knn_type, user_based, mink=sel.MINK, extra=extra)
        shards = _shards(uu, ii, r, "msd", knn_type, user_based, "cyclic", 2, mink=sel.MINK, extra=extra)
        for e in (full, *shards):
            e._h.set_k(256, sel.MINK)
        side = "left" if user_based else "right"
        q = full.Data.convert_users(left if user_based else items)
        ref = ob.KNN(sim="msd", knn_type=knn_type, user_based=user_based, k=256, min_k=sel.MINK, n_jobs=8,
                     tie_policy="canonical").fit(ob.TrainSet(uu, ii, r))
        _check(shards, full, side, q, (10,), score_all(ref, uu, ii, user_based, side, q))
        _close(full, *shards)


# ---- edge cases ----
def test_query_that_rated_every_target():
    u = np.array([0] * 6 + [1, 1, 2, 2, 3], dtype=np.int64)
    i = np.array([0, 1, 2, 3, 4, 5, 0, 1, 2, 3, 4], dtype=np.int64)
    r = np.array([1, 2, 3, 4, 5, 1, 2, 3, 4, 5, 1], dtype=np.float64)
    for user_based in (True, False):
        full = trg._fit(u, i, r, "msd", "basic", user_based, extra={"simPath": "stream"})
        shards = _shards(u, i, r, "msd", "basic", user_based, "cyclic", 2, extra={"simPath": "stream"})
        side = "left" if user_based else "right"
        _check(shards, full, side, [0, 1, -1], (3, 8))
        _close(full, *shards)


def test_batches_and_empty_calls(ml100k, monkeypatch):
    import torch

    u, i, r = split(ml100k["u1_base"])
    for user_based in (True, False):
        full = trg._fit(u, i, r, "pearson", "centered", user_based, extra={"simPath": "stream"})
        shards = _shards(u, i, r, "pearson", "centered", user_based, "cyclic", 2, extra={"simPath": "stream"})
        side = "left" if user_based else "right"
        q = np.concatenate([np.arange(0, 943, 7), [-1]])
        monkeypatch.setenv("RS_KNN_REC_BATCH", "3")
        _check(shards, full, side, q, (20,))
        monkeypatch.delenv("RS_KNN_REC_BATCH")
        d = torch.empty(1, dtype=torch.int32, device="cuda")
        for s in shards:                                  # n = 0: nothing to do
            s._h.recommend_sharded_device(side, d.data_ptr(), 0, 5, d.data_ptr(), d.data_ptr())
            s._h.score_all_sharded_device(side, d.data_ptr(), 0, d.data_ptr())
        _close(full, *shards)


# ---- refusals ----
def test_refusals(ml100k):
    import torch

    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    d_q = torch.zeros(4, dtype=torch.int32, device="cuda")
    d_i = torch.empty(4 * 513, dtype=torch.int32, device="cuda")
    d_s = torch.empty(4 * 1682, dtype=torch.float64, device="cuda")

    def refused(h, n=1, n_top=5, side="left"):
        with pytest.raises(RuntimeError):
            h.recommend_sharded_device(side, d_q.data_ptr(), n, n_top, d_i.data_ptr(), d_s.data_ptr())
        if n_top == 5:
            with pytest.raises(RuntimeError):
                h.score_all_sharded_device(side, d_q.data_ptr(), n, d_s.data_ptr())

    # cyclic shards before the mirror step
    shards = [trg._fit(u, i, r, "msd", "basic", True, extra={"shardCount": 2, "shardIndex": s}) for s in range(2)]
    for s in shards:
        refused(s._h)
    for s in shards:
        s._h.synchronize()
    for s in shards:
        s._h.peer_import_local([x._h for x in shards])
        s._h.mirror()
    h = shards[0]._h
    for n_top in (0, 513):
        refused(h, n_top=n_top)
    for n in (-1, 1 << 31):
        refused(h, n=n)
    with pytest.raises(RuntimeError):                     # the plain entry points keep refusing shards
        h.recommend("left", [0], 5)
    with pytest.raises(RuntimeError):
        h.score_all("left", [0])
    h.set_k(257, 1)
    refused(h)
    _close(*shards)
    # not a row shard, top-k lists, Slope One
    full = trg._fit(u, i, r, "msd", "basic", True, extra={"simPath": "stream"})
    refused(full._h)
    full.Close()
    topk = trg._fit(u, i, r, "msd", "basic", True, extra={"simPath": "stream", "store": "topk", "topk": 40,
                                                          "rowBegin": 0, "rowEnd": 128})
    refused(topk._h)
    topk.Close()
    so = rs.NewSlopeOne(rs.Parameters({"rowBegin": 0, "rowEnd": 128}))
    so.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    refused(so._h, side="right")
    so.Close()


# ---- ShardedKNN over NCCL, two GPUs ----
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


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
    users = np.concatenate([np.unique(u)[::5], [10 ** 9]])          # the last one is unknown
    for user_based in (True, False):
        params = {"sim": rs.Pearson, "userBased": user_based, "k": 40}
        est = rs.shard.ShardedKNN(rs.NewKNNWithMean(rs.Parameters(params)))
        est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
        items, scores = est.Recommend(users, 25)
        rows = est.ScoreAll(users)
        if rank == 0:
            one = rs.NewKNNWithMean(rs.Parameters(params))
            one.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
            wi, ws = one.Recommend(users, 25)
            assert np.array_equal(items, wi) and same_bits(scores, ws), user_based
            assert same_bits(rows, one.ScoreAll(users)), user_based
            one.Close()
        est.Close()
    if rank == 0:
        (Path(out_dir) / "ok").write_text("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_knn_two_gpus(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok").read_text() == "ok"
