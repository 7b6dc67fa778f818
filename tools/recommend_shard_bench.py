"""Top-N recommendation on cyclic row shards: the per-shard call and the union of the partial lists.

Workload: the ML-20M item shape (bench.py ml20m_item_pearson_k40), centered Pearson, k = 40, the 1,024 seeded uniform
users of tools/recommend_bench.py, n_top 100 (right queries: each shard scores the items it owns).  On one GPU the
matrix is fitted as 1, 2, 4 and 8 cyclic shards, wired with rs_knn_peer_import_local + rs_knn_mirror; for each count
the script times rs_knn_recommend_sharded_device on every shard (shard 0 and the slowest are reported) and the union
of the partial lists (shard.union_recommend_device), and checks that the united lists equal rs_knn_recommend_device of
one full handle bit for bit.  Count 1 is that full handle's call.  CUDA events on the current stream, median of
--repeats after a warm-up, the L2 overwritten (a 512 MiB write) before every timed repeat, outside the window.
With 2 GPUs visible, one NCCL end-to-end ShardedKNN.Recommend (2 ranks) is timed too.
Usage: python tools/recommend_shard_bench.py [--repeats 5] [--quick]"""
import argparse
import json
import os
import socket
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

N_TOP = 100
NQ = 1024


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def make_train(quick):
    import bench
    import recommend_sys_b200 as rs

    if quick:
        return rs.NewTrainSet(rs.core.synth_ratings(2000, 1500, 200_000, 0x5EED0042))
    return bench.make_data("ml20m_item_pearson_k40")[0]


def queries_of(train):
    rng = np.random.RandomState(0x5EED)
    return np.sort(rng.choice(train.UserCount, NQ, replace=False)).astype(np.int32)


def timed(fn, repeats, torch, flush):
    fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(repeats):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        t.append(a.elapsed_time(b))
    return float(np.median(t))


def new_knn(rs, **extra):
    return rs.NewKNNWithMean(rs.Parameters(dict({"sim": rs.Pearson, "userBased": False, "k": 40}, **extra)))


def one_gpu(args, torch, rs):
    from recommend_sys_b200.shard import union_recommend_device

    train = make_train(args.quick)
    q = queries_of(train)
    dq = torch.from_numpy(q).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    full = new_knn(rs)
    full.Fit(train)
    full._h.set_stream(stream)
    wi = torch.empty((NQ, N_TOP), dtype=torch.int32, device="cuda")
    ws = torch.empty((NQ, N_TOP), dtype=torch.float64, device="cuda")
    t_full = timed(lambda: full._h.recommend_device("right", dq.data_ptr(), NQ, N_TOP, wi.data_ptr(), ws.data_ptr()),
                   args.repeats, torch, flush)
    want_i, want_s = wi.cpu().numpy(), ws.cpu().numpy()
    full.Close()
    rows = [{"shards": 1, "rows_local": int(train.ItemCount), "shard0_ms": round(t_full, 3),
             "slowest_shard_ms": round(t_full, 3), "union_ms": 0.0, "identical_lists": True}]
    print(json.dumps(rows[0]), flush=True)
    for count in (2, 4, 8):
        shards = []
        for s in range(count):
            e = new_knn(rs, shardCount=count, shardIndex=s)
            e.Fit(train)
            shards.append(e)
        for e in shards:
            e._h.synchronize()
        for e in shards:
            e._h.peer_import_local([x._h for x in shards])
            e._h.mirror()
            e._h.set_stream(stream)
        ai = torch.empty((count, NQ, N_TOP), dtype=torch.int32, device="cuda")
        as_ = torch.empty((count, NQ, N_TOP), dtype=torch.float64, device="cuda")
        t_sh = []
        for j, e in enumerate(shards):
            t_sh.append(timed(lambda: e._h.recommend_sharded_device("right", dq.data_ptr(), NQ, N_TOP, ai[j].data_ptr(),
                                                                   as_[j].data_ptr()), args.repeats, torch, flush))
        out = {}

        def unite():
            out["r"] = union_recommend_device(ai, as_)

        t_u = timed(unite, args.repeats, torch, flush)
        gi, gs = out["r"][0].cpu().numpy(), out["r"][1].cpu().numpy()
        same = (np.array_equal(gi, want_i) and np.array_equal(np.isnan(gs), np.isnan(want_s))
                and np.array_equal(gs[~np.isnan(gs)].view(np.uint64), want_s[~np.isnan(want_s)].view(np.uint64)))
        row = {"shards": count, "rows_local": int(shards[0]._h.owned_rows().size), "shard0_ms": round(t_sh[0], 3),
               "slowest_shard_ms": round(max(t_sh), 3), "union_ms": round(t_u, 3),
               "union_share": round(t_u / (max(t_sh) + t_u), 4), "identical_lists": bool(same)}
        print(json.dumps(row), flush=True)
        rows.append(row)
        for e in shards:
            e.Close()
        assert same, f"{count} shards: the united lists differ from the full handle's"
    return rows


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, quick, repeats, out_path):
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist

    import recommend_sys_b200 as rs

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    train = make_train(quick)
    users = train.Users[np.unique(train.innerUsers, return_index=True)[1]][queries_of(train)]
    est = rs.shard.ShardedKNN(new_knn(rs))
    est.Fit(train)
    est.Recommend(users, N_TOP)
    t = []
    for _ in range(repeats):
        dist.barrier()
        t0 = time.perf_counter()
        est.Recommend(users, N_TOP)        # returns host arrays: ends in a device synchronise
        t.append((time.perf_counter() - t0) * 1e3)
    if rank == 0:
        Path(out_path).write_text(json.dumps({"nccl_ranks": world, "sharded_knn_recommend_ms": round(float(np.median(t)), 3)}))
    est.Close()
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    import torch

    import recommend_sys_b200 as rs

    if not torch.cuda.is_available():
        raise SystemExit("recommend_shard_bench.py needs a CUDA device")
    print(json.dumps({"card": card()}), flush=True)
    one_gpu(args, torch, rs)
    if torch.cuda.device_count() >= 2:
        import tempfile

        import torch.multiprocessing as mp

        with tempfile.TemporaryDirectory() as d:
            out = os.path.join(d, "nccl.json")
            mp.spawn(_nccl_worker, args=(2, _free_port(), args.quick, args.repeats, out), nprocs=2, join=True)
            print(Path(out).read_text(), flush=True)
    else:
        print(json.dumps({"nccl_ranks": 2, "sharded_knn_recommend_ms": "not measured (fewer than 2 GPUs)"}), flush=True)
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
