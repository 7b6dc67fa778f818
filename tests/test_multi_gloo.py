"""N>1 host logic on CPU: world_size 2 over gloo (no GPU).  Each rank owns a row shard, computes
its neighbour lists and its share of the predictions with the ORACLE standing in for the device
(the sharding / all-gather plumbing is what is under test), and the gathered result must equal
the single-shard result."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import load_ml100k

ROOT = Path(__file__).resolve().parent.parent


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist

    from oracle import binding as ob
    from recommend_sys_b200.shard import allgather_predictions, allgather_topk, shard_rows

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = load_ml100k()
    tr = g["u1_base"][:30000]
    te = g["u1_test"][:3000]
    ts = ob.TrainSet(tr[:, 0], tr[:, 1], tr[:, 2].astype(float))
    n = ts.user_count
    b, e = shard_rows(n, world, rank, align=16)
    knn = ob.KNN(sim="msd", k=10, user_based=True).fit(ts, rows=(b, e))   # this rank's rows only
    idx, sim = knn.topk(10, b, e)
    all_i, all_s = allgather_topk(torch.from_numpy(idx), torch.from_numpy(sim), n, 10, align=16)
    # predictions: each test pair goes to the owner of its left row
    L = ob.lib()
    left = np.array([L.or_trainset_convert_user(ts.h, int(u)) for u in te[:, 0]])
    mine = np.where(((left >= b) & (left < e)) | ((left < 0) & (rank == 0)))[0]
    pred = knn.predict_batch(te[mine, 0], te[mine, 1])
    counts = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(counts, torch.tensor([len(mine)]))
    counts = [int(c) for c in counts]
    gathered = allgather_predictions(torch.from_numpy(pred), counts)
    if rank == 0:
        full = ob.KNN(sim="msd", k=10, user_based=True).fit(ts)
        wi, ws = full.topk(10)
        assert np.array_equal(all_i.numpy(), wi)
        assert np.array_equal(np.nan_to_num(all_s.numpy()), np.nan_to_num(ws))
        want = full.predict_batch(te[:, 0], te[:, 1])
        # rebuild the order: rank r's predictions are for its `mine` indices (recomputed here)
        got = np.full(len(te), np.nan)
        off = 0
        for r in range(world):
            rb, re = shard_rows(n, world, r, align=16)
            m = np.where(((left >= rb) & (left < re)) | ((left < 0) & (r == 0)))[0]
            got[m] = gathered.numpy()[off:off + len(m)]
            off += len(m)
        assert np.array_equal(np.nan_to_num(got), np.nan_to_num(want))
        (Path(out_dir) / "ok").write_text("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_shard_allgather(tmp_path):
    import torch.multiprocessing as mp

    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok").read_text() == "ok"


def _topk_canonical(ids, sims, k):
    """Top k of (id, sim) candidates, similarity desc then id asc; NaN excluded; padded with -1 / NaN."""
    ok = ~np.isnan(sims)
    ids, sims = ids[ok], sims[ok]
    order = np.lexsort((ids, -(sims + 0.0)))[:k]
    oi = np.full(k, -1, dtype=np.int32)
    os_ = np.full(k, np.nan)
    oi[:len(order)] = ids[order]
    os_[:len(order)] = sims[order]
    return oi, os_


def _worker_symmetric(rank, world, port, out_dir):
    """Symmetric-slab sharding (rs_knn_params.shard_count): rank r owns the slabs r, r+world, ... and of
    each only the pairs right of the diagonal; every pair feeds both rows' PARTIAL lists; one
    all-gather + union gives the final lists.  The oracle stands in for the device."""
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist

    from oracle import binding as ob
    from recommend_sys_b200.shard import allgather_partial_topk, slab_owner

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = load_ml100k()
    tr = g["u1_base"][:20000]
    ts = ob.TrainSet(tr[:, 0], tr[:, 1], tr[:, 2].astype(float))
    full = ob.KNN(sim="msd", k=10, user_based=True).fit(ts)
    S = full.sims()
    n, k, m = S.shape[0], 10, 64
    cand = [([], []) for _ in range(n)]
    for slab in range((n + m - 1) // m):
        if slab_owner(slab, world) != rank:
            continue
        for i in range(slab * m, min(n, slab * m + m)):
            for j in range(i + 1, n):
                cand[i][0].append(j); cand[i][1].append(S[i, j])
                cand[j][0].append(i); cand[j][1].append(S[i, j])
    part_i = np.full((n, k), -1, dtype=np.int32)
    part_s = np.full((n, k), np.nan)
    for r in range(n):
        part_i[r], part_s[r] = _topk_canonical(np.array(cand[r][0], dtype=np.int32), np.array(cand[r][1]), k)
    all_i, all_s = allgather_partial_topk(torch.from_numpy(part_i), torch.from_numpy(part_s))
    assert tuple(all_i.shape) == (world, n, k)
    if rank == 0:
        wi, ws = full.topk(k)
        ai, as_ = all_i.numpy(), all_s.numpy()
        for r in range(n):
            ids = ai[:, r, :].reshape(-1)
            keep = ids >= 0
            assert len(np.unique(ids[keep])) == keep.sum()          # every pair in exactly one partial list
            gi, gs = _topk_canonical(ids[keep], as_[:, r, :].reshape(-1)[keep], k)
            assert np.array_equal(gi, wi[r]) and np.array_equal(np.nan_to_num(gs), np.nan_to_num(ws[r]))
        (Path(out_dir) / "ok_sym").write_text("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_symmetric_slabs(tmp_path):
    import torch.multiprocessing as mp

    port = _free_port()
    mp.spawn(_worker_symmetric, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok_sym").read_text() == "ok"


def _worker_cyclic(rank, world, port, out_dir):
    """Cyclic row shards (RS_STORE_MATRIX, shard_count >= 2; ShardedKNN): rows dealt in blocks of 32, every rank
    computes ONE triangle of its rows, the other triangle is the transpose of cells other ranks computed
    (here exchanged with an all-gather, on the device pulled from peer memory), test pairs are routed to the
    owner of their left row and the predictions all-gathered.  The oracle stands in for the device."""
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist

    import recommend_sys_b200 as rs
    from oracle import binding as ob
    from recommend_sys_b200.shard import allgather_predictions, route_pairs

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = load_ml100k()
    tr = g["u1_base"][:30000]
    te = g["u1_test"][:3000]
    ts = ob.TrainSet(tr[:, 0], tr[:, 1], tr[:, 2].astype(float))
    full = ob.KNN(sim="pearson", knn_type="centered", k=10, user_based=True).fit(ts)
    S = full.sims()
    n = S.shape[0]
    rows = rs.core.cyclic_rows(n, world, rank)
    assert np.array_equal(rs.core.cyclic_owner(rows, world), np.full(len(rows), rank))
    # this rank's lower triangle only (what the device kernel leaves before rs_knn_mirror)
    mine = np.full((len(rows), n), np.nan)
    for li, i in enumerate(rows):
        mine[li, :i] = S[i, :i]
    # exchange: every rank publishes its triangle; a rank fills (i, j > i) from the owner of row j
    sizes = [len(rs.core.cyclic_rows(n, world, r)) for r in range(world)]
    pad = torch.full((max(sizes), n), float("nan"), dtype=torch.float64)     # shard sizes differ by up to 32 rows
    pad[: len(rows)] = torch.from_numpy(mine)
    allp = [torch.empty((max(sizes), n), dtype=torch.float64) for _ in range(world)]
    dist.all_gather(allp, pad)
    parts = [allp[r][: sizes[r]] for r in range(world)]
    local_of = {}
    for r in range(world):
        for li, i in enumerate(rs.core.cyclic_rows(n, world, r)):
            local_of[int(i)] = (r, li)
    for li, i in enumerate(rows):
        for j in range(int(i) + 1, n):
            r, lj = local_of[j]
            mine[li, j] = parts[r][lj, i]
    assert np.array_equal(np.nan_to_num(mine), np.nan_to_num(S[rows]))
    # predictions: routed to the owner of the left row, cold-start pairs spread evenly, all-gathered
    L = ob.lib()
    left = np.array([L.or_trainset_convert_user(ts.h, int(u)) for u in te[:, 0]])
    owner = route_pairs(left, world)
    assert ((left < 0) | (owner == rs.core.cyclic_owner(np.maximum(left, 0), world))).all()
    order = np.argsort(owner, kind="stable")
    counts = np.bincount(owner, minlength=world).tolist()
    sel = order[sum(counts[:rank]): sum(counts[:rank + 1])]
    pred = full.predict_batch(te[sel, 0], te[sel, 1])
    gathered = allgather_predictions(torch.from_numpy(pred), counts).numpy()
    out = np.empty(len(te))
    out[order] = gathered
    want = full.predict_batch(te[:, 0], te[:, 1])
    assert np.array_equal(np.nan_to_num(out), np.nan_to_num(want))
    # the all-reduce form (ShardedKNN.PredictBatch): own pairs answered, +0.0 elsewhere, int64 sum of the bit patterns
    part = np.zeros(len(te))
    part[sel] = pred
    acc = torch.from_numpy(part.view(np.int64).copy())
    dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    got = acc.numpy().view(np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(got[~np.isnan(got)].view(np.int64),
                                                                             want[~np.isnan(want)].view(np.int64))
    if rank == 0:
        (Path(out_dir) / "ok_cyc").write_text("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_cyclic_row_shards(tmp_path):
    import torch.multiprocessing as mp

    port = _free_port()
    mp.spawn(_worker_cyclic, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok_cyc").read_text() == "ok"
