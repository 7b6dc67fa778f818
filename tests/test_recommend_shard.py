"""Top-N recommendation on row shards, host side: the ownership rule and the union of partial lists over gloo (the
oracle stands in for the device), the local -> global row map of cyclic shards, and the tree union of
shard.union_recommend_device."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import load_ml100k
from recommend_ref import rank_rows, same_bits, score_all

ROOT = Path(__file__).resolve().parent.parent
CYC_B = 32


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _np_union(all_i, all_s):
    """Numpy restatement of rs_knn_topk_union_device: every listed entry of every list, ranked by (score desc, id
    asc) with +-0 tied, the best k kept, unused slots -1 / NaN."""
    import torch

    ai, as_ = np.asarray(all_i), np.asarray(all_s)
    n_lists, n, k = ai.shape
    assert n_lists * k <= 2048
    out_i = np.full((n, k), -1, dtype=np.int32)
    out_s = np.full((n, k), np.nan)
    for r in range(n):
        ids, s = ai[:, r].ravel(), as_[:, r].ravel()
        keep = ids >= 0
        ids, s = ids[keep], s[keep]
        assert len(np.unique(ids)) == len(ids)           # every target is in at most one partial list
        order = np.lexsort((ids, -(s + 0.0)))[:k]
        out_i[r, :len(order)] = ids[order]
        out_s[r, :len(order)] = s[order]
    return torch.from_numpy(out_i), torch.from_numpy(out_s)


def _owned(ids, count, index):
    return (np.asarray(ids) // CYC_B) % count == index


def _partial_lists(rows, side, queries, count, index, n_top):
    """The partial lists of shard `index` of `count` cyclic shards under the ownership rule of
    rs_knn_recommend_sharded_device, from the full score rows."""
    rows = rows.copy()
    if side == "right":                                   # the shard lists only the targets it owns
        rows[:, ~_owned(np.arange(rows.shape[1]), count, index)] = np.nan
        return rank_rows(rows, n_top)
    answer = _owned(np.maximum(queries, 0), count, index)   # -1: the owner of row 0
    ids, top = rank_rows(rows, n_top)
    ids[~answer] = -1
    top[~answer] = np.nan
    return ids, top


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch
    import torch.distributed as dist

    from oracle import binding as ob
    from recommend_sys_b200.shard import allgather_partial_topk, union_recommend_device

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    tr = load_ml100k()["u1_base"][:20000]
    u, i, r = tr[:, 0], tr[:, 1], tr[:, 2].astype(np.float64)
    for user_based, side in ((False, "right"), (True, "left")):
        ref = ob.KNN(sim="msd", knn_type="basic", user_based=user_based, k=20, n_jobs=4,
                     tie_policy="canonical").fit(ob.TrainSet(u, i, r))
        queries = np.concatenate([np.arange(0, 200, 3), [-1, -1]])
        rows = score_all(ref, u, i, user_based, side, queries)
        for n_top in (1, 10, 300):
            ids, top = _partial_lists(rows, side, queries, world, rank, n_top)
            all_i, all_s = allgather_partial_topk(torch.from_numpy(ids), torch.from_numpy(top))
            if side == "left":                            # every list comes from exactly one shard
                assert ((all_i[:, :, 0] >= 0).sum(0) <= 1).all()
            got_i, got_s = union_recommend_device(all_i, all_s, unite=_np_union)
            want_i, want_s = rank_rows(rows, n_top)
            assert np.array_equal(got_i.numpy(), want_i), (side, n_top)
            assert same_bits(got_s.numpy(), want_s)
    if rank == 0:
        (Path(out_dir) / "ok").write_text("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_partial_lists_unite(tmp_path):
    import torch.multiprocessing as mp

    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok").read_text() == "ok"


@pytest.mark.parametrize("n", [1, 31, 32, 33, 943, 1682, 4100])
@pytest.mark.parametrize("count", [2, 3, 5, 8])
def test_cyclic_local_to_global(n, count):
    """rs_cyc_global (csrc/common.cuh) restated: strictly increasing over a shard's local rows, the inverse of
    rs_cyc_local, and the shard's rows in storage order (core.cyclic_rows)."""
    import recommend_sys_b200 as rs

    seen = []
    for index in range(count):
        rows = rs.core.cyclic_rows(n, count, index)
        loc = np.arange(len(rows))
        glob = ((loc // CYC_B) * count + index) * CYC_B + loc % CYC_B
        assert np.array_equal(glob, rows)
        assert (np.diff(glob) > 0).all()
        assert np.array_equal((glob // (CYC_B * count)) * CYC_B + glob % CYC_B, loc)     # rs_cyc_local
        seen.append(glob)
    assert np.array_equal(np.sort(np.concatenate(seen)), np.arange(n))


@pytest.mark.parametrize("n_lists", [1, 2, 4, 5, 8, 17])
@pytest.mark.parametrize("n_top", [1, 10, 100, 512])
def test_tree_union(n_lists, n_top):
    """union_recommend_device unites any number of partial lists with calls of at most 2048 entries per row, and the
    result is the ranking of all entries."""
    import torch

    from recommend_sys_b200.shard import union_recommend_device

    rng = np.random.RandomState(n_lists * 1000 + n_top)
    n_rows, n_targets = 3, 6000
    scores = rng.choice([-1.5, -0.0, 0.0, 0.5, 2.0, np.inf, -np.inf, np.nan], size=(n_rows, n_targets))
    scores[:, ::7] = rng.randn(n_rows, len(range(0, n_targets, 7)))
    owner = rng.randint(0, n_lists, n_targets)
    all_i = np.empty((n_lists, n_rows, n_top), np.int32)
    all_s = np.empty((n_lists, n_rows, n_top))
    for s in range(n_lists):
        part = np.where(owner == s, scores, np.nan)
        all_i[s], all_s[s] = rank_rows(part, n_top)
    calls = []

    def unite(ai, as_):
        calls.append(ai.shape[0])
        assert ai.shape[0] * n_top <= 2048
        return _np_union(ai, as_)

    got_i, got_s = union_recommend_device(torch.from_numpy(all_i), torch.from_numpy(all_s), unite=unite)
    want_i, want_s = rank_rows(scores, n_top)
    assert np.array_equal(got_i.numpy(), want_i) and same_bits(got_s.numpy(), want_s)
    group = 2048 // n_top
    assert calls[0] == min(n_lists, group)
    assert len(calls) >= -(-n_lists // group)
