"""Top-N recommendation on the device against the composition a caller would otherwise build from Predict.

  new path     rs_knn_recommend_device: score every target of each query, rated targets excluded, top N.
  composition  rs_knn_predict_batch_device over all Q x n_targets pairs, the rated targets set to NaN, and a top N
               under the same rule (score desc, target id asc, NaN never listed) with two stable torch sorts.

Both are timed with CUDA events on the handle's stream after a warm-up; the L2 is overwritten (a 512 MiB write)
before every timed repeat, outside the timed window.  Both must produce identical lists.  Runs:
  item-based  the ML-20M item shape (bench.py ml20m_item_pearson_k40), centered Pearson, k = 40, 1,024 queries:
              a seeded uniform sample of users and the 1,024 users with the most training ratings, n_top 10 / 100;
  user-based  the ML-1M user shape, MSD basic, all 6,040 users, n_top 10.
Usage: python tools/recommend_bench.py [--repeats 5]"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def composition(h, torch, side, q, n_targets, n_top, rated_flat, bufs):
    """Predict every pair, NaN the rated ones, top N by (score desc, id asc) via stable sorts."""
    dl, dr, out = bufs
    h.predict_batch_device(dl.data_ptr(), dr.data_ptr(), dl.numel(), out.data_ptr())
    s = out.view(len(q), n_targets)
    s.view(-1)[rated_flat] = float("nan")
    nan = torch.isnan(s)
    key = torch.where(nan, torch.full_like(s, float("-inf")), s + 0.0)      # -0.0 and +0.0 share a key
    o1 = torch.sort(key, dim=1, descending=True, stable=True).indices
    o2 = torch.sort(torch.gather(nan, 1, o1).to(torch.int8), dim=1, stable=True).indices
    ids = torch.gather(o1, 1, o2)[:, :n_top]
    sc = torch.gather(s, 1, ids)
    ok = ~torch.isnan(sc)
    return torch.where(ok, ids, -1).to(torch.int32), sc


def run(name, est, side, queries, n_tops, repeats, torch):
    rs_h = est._h
    stream = torch.cuda.current_stream()
    rs_h.set_stream(stream.cuda_stream)
    n_targets = rs_h.n_left if side == "right" else rs_h.n_right
    nq = len(queries)
    dq = torch.tensor(queries, dtype=torch.int32, device="cuda")
    qq = np.repeat(queries.astype(np.int32), n_targets)
    tt = np.tile(np.arange(n_targets, dtype=np.int32), nq)
    l, r = (qq, tt) if side == "left" else (tt, qq)
    bufs = (torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda(), torch.empty(nq * n_targets, dtype=torch.float64,
                                                                                  device="cuda"))
    # rated targets of each query, flat into [nq][n_targets]
    d = est.Data
    lu, ri = (d.innerUsers, d.innerItems) if est._userBased else (d.innerItems, d.innerUsers)
    qs, ts = (lu, ri) if side == "left" else (ri, lu)
    pos = {int(v): b for b, v in enumerate(queries.tolist())}
    rows = [[] for _ in range(nq)]
    for a, t in zip(qs.tolist(), ts.tolist()):
        b = pos.get(a)
        if b is not None:
            rows[b].append(b * n_targets + t)
    rated_flat = torch.tensor(np.concatenate([np.asarray(x, dtype=np.int64) for x in rows]), device="cuda")
    if side == "right":
        cnt = np.bincount(d.innerUsers if not est._userBased else d.innerItems, minlength=rs_h.n_right)
        visits = float(cnt[queries].sum()) * n_targets      # |R(q)| candidates for every target
        matrix_bytes = visits * 8                           # S[j][t] for j in R(q), every target t
    else:
        visits = float(len(d.innerUsers)) * nq              # every target's raters, once per query
        matrix_bytes = float(nq) * rs_h.n_left * 8          # the row S[q][.] of each query (gathered from L2)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    res = []
    for n_top in n_tops:
        ids = torch.empty((nq, n_top), dtype=torch.int32, device="cuda")
        sc = torch.empty((nq, n_top), dtype=torch.float64, device="cuda")

        def new():
            rs_h.recommend_device(side, dq.data_ptr(), nq, n_top, ids.data_ptr(), sc.data_ptr())
            return ids, sc

        def old():
            return composition(rs_h, torch, side, queries, n_targets, n_top, rated_flat, bufs)

        times = {}
        outs = {}
        for label, fn in (("new", new), ("composition", old)):
            fn()
            torch.cuda.synchronize()
            t = []
            for _ in range(repeats):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                o = fn()
                b.record(stream)
                torch.cuda.synchronize()
                t.append(a.elapsed_time(b))
            times[label] = float(np.median(t))
            outs[label] = (o[0].cpu().numpy().copy(), o[1].cpu().numpy().copy())
        ni, ns = outs["new"]
        ci, cs = outs["composition"]
        nn, cn = np.isnan(ns), np.isnan(cs)
        same = (np.array_equal(ni, ci) and np.array_equal(nn, cn)
                and np.array_equal(ns[~nn].view(np.uint64), cs[~cn].view(np.uint64)))
        row = {"run": name, "side": side, "queries": nq, "n_targets": n_targets, "n_top": n_top,
               "new_ms": round(times["new"], 3), "composition_ms": round(times["composition"], 3),
               "speedup": round(times["composition"] / times["new"], 2), "identical_lists": bool(same),
               "candidate_visits": visits, "matrix_bytes_new": matrix_bytes,
               "matrix_rate_GBps": round(matrix_bytes / (times["new"] * 1e-3) / 1e9, 1)}
        print(json.dumps(row), flush=True)
        res.append(row)
        assert same, f"{name} n_top={n_top}: the new path and the composition list different targets"
    rs_h.set_stream(0, use_own=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    import torch

    import bench
    import recommend_sys_b200 as rs

    if not torch.cuda.is_available():
        raise SystemExit("recommend_bench.py needs a CUDA device")
    print(json.dumps({"card": card()}), flush=True)
    if args.quick:
        data = rs.core.synth_ratings(2000, 1500, 200_000, 0x5EED0042)
        train = rs.NewTrainSet(data)
    else:
        train, _ = bench.make_data("ml20m_item_pearson_k40")
    est = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False, "k": 40}))
    est.Fit(train)
    est._h.synchronize()
    cnt = np.bincount(train.innerUsers, minlength=train.UserCount)
    rng = np.random.RandomState(0x5EED)
    nq = 1024
    uniform = np.sort(rng.choice(train.UserCount, nq, replace=False))
    heavy = np.sort(np.argsort(-cnt, kind="stable")[:nq])
    run("ml20m_item_uniform", est, "right", uniform, (10, 100), args.repeats, torch)
    run("ml20m_item_heaviest", est, "right", heavy, (10, 100), args.repeats, torch)
    est.Close()
    if args.quick:
        data = rs.core.synth_ratings(800, 600, 60_000, 0x5EED0043)
    else:
        data = rs.core.synth_ratings(6040, 3706, 1_000_000, 0x5EED0044)
    train = rs.NewTrainSet(data)
    est = rs.NewKNN(rs.Parameters({"sim": rs.MSD, "userBased": True, "k": 40}))
    est.Fit(train)
    est._h.synchronize()
    run("ml1m_user_msd", est, "left", np.arange(train.UserCount), (10,), args.repeats, torch)
    est.Close()
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
