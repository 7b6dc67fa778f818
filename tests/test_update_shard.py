"""ShardedKNN.Update, host side, over gloo with two ranks and a fake handle in place of the device: the same refusal on
every rank raises that error on every rank and leaves the estimator as it was; a split outcome raises on every rank
and every later call refuses until the next Fit; after a success Data and GlobalMean are TrainSet.Extend's."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import load_ml100k, split

ROOT = Path(__file__).resolve().parent.parent


class _FakeHandle:
    """Stands in for a mirrored cyclic shard: records each update and answers with the planned return code."""

    def __init__(self, codes):
        self.codes = list(codes)
        self.calls = []

    def update_sharded_device(self, d_left, d_right, d_rating, nnz, n_left, n_right, global_mean):
        from recommend_sys_b200 import core

        self.calls.append((nnz, n_left, n_right, global_mean))
        code = self.codes.pop(0)
        if code != 0:
            raise core.RsError(code, "planned")

    def close(self):
        pass


def _estimator(rs, train, codes):
    import torch

    from recommend_sys_b200.shard import ShardedKNN

    class CpuShardedKNN(ShardedKNN):
        def _device(self):
            return torch.device("cpu")

    knn = rs.NewKNN(rs.Parameters({"sim": rs.MSD, "userBased": True}))
    knn.Data, knn.GlobalMean, knn._userBased = train, train.GlobalMean, True
    knn._h = _FakeHandle(codes)
    return CpuShardedKNN(knn)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch.distributed as dist

    import recommend_sys_b200 as rs
    from recommend_sys_b200 import core

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    u, i, r = split(load_ml100k()["u1_base"])
    m = len(r) - 500
    train = rs.NewTrainSet(rs.NewRawSet(u[:m], i[:m], r[:m]))
    add = rs.NewRawSet(np.concatenate([u[m:], [5001]]), np.concatenate([i[m:], [9001]]),
                       np.concatenate([r[m:], [2.0]]))
    want = train.Extend(add)

    # the same refusal on both ranks: that error on both, the estimator unchanged, and the next Update goes through
    est = _estimator(rs, train, [-5, 0])
    with pytest.raises(core.RsError) as e:
        est.Update(add)
    assert e.value.code == -5 and "planned" in str(e.value)
    assert est.knn.Data is train and est.knn.GlobalMean == train.GlobalMean
    est.Update(add)
    got = est.knn.Data
    assert got.UserCount == want.UserCount and got.ItemCount == want.ItemCount
    assert np.array_equal(got.innerUsers, want.innerUsers) and np.array_equal(got.innerItems, want.innerItems)
    assert np.array_equal(got.Ratings.view(np.uint64), want.Ratings.view(np.uint64))
    assert np.float64(est.knn.GlobalMean).view(np.uint64) == np.float64(want.GlobalMean).view(np.uint64)
    assert est.knn._h.calls[-1] == (len(r) - m + 1, want.UserCount, want.ItemCount, want.GlobalMean)

    # a split outcome: rank 0 fails (out of memory), rank 1 succeeds; both raise, and every later call refuses
    est = _estimator(rs, train, [-4 if rank == 0 else 0])
    with pytest.raises(core.RsError) as e:
        est.Update(add)
    assert e.value.code == -4 and "disagree" in str(e.value)
    for call in (lambda: est.Update(add), lambda: est.PredictBatch(np.array([1]), np.array([1])),
                 lambda: est.Recommend(np.array([1]), 5), lambda: est.ScoreAll(np.array([1]))):
        with pytest.raises(RuntimeError, match="Fit again"):
            call()
    assert est.knn._h.calls and len(est.knn._h.calls) == 1          # nothing reached the handle after the split
    if rank == 0:
        (Path(out_dir) / "ok").write_text("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_update_outcomes(tmp_path):
    import torch.multiprocessing as mp

    from test_recommend_shard import _free_port

    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok").read_text() == "ok"
