"""Recommendation for queries given as rating lists (rs_knn_recommend_given_device) against the same users asked by id
(rs_knn_recommend_device): the lists are the users' own training ratings, so both must list the same targets.

Both calls are timed with CUDA events on the handle's stream after a warm-up, alternated repeat by repeat; the L2 is
overwritten (a 512 MiB write) before every timed call, outside the timed window.  Runs:
  item-based  the ML-20M item shape (bench.py ml20m_item_pearson_k40), centered Pearson, k = 40, the 1,024 uniform
              users of tools/recommend_bench.py, n_top 10: the same kernel on the same candidates, expected equal;
  user-based  the ML-1M user shape, MSD basic, k = 40, all 6,040 users, n_top 10: the given call computes each list's
              similarity row first (given_sims_kernel).  Its time alone comes from a torch.profiler pass of its own
              (CUDA activities), and its rate is counted in (list entry, rater) updates: sum over the lists' entries c
              of |R(c)|.
Usage: python tools/recommend_given_bench.py [--repeats 7] [--quick]"""
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
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def own_lists(est, queries):
    """The queries' own training ratings as lists of inner item ids in dataset order (ptr, ids, vals)."""
    d = est.Data
    pos = np.full(d.UserCount, -1, dtype=np.int64)
    pos[queries] = np.arange(len(queries))
    b = pos[d.innerUsers]
    keep = b >= 0
    order = np.argsort(b[keep], kind="stable")
    ids = d.innerItems[keep][order].astype(np.int32)
    vals = d.Ratings[keep][order].astype(np.float64)
    ptr = np.zeros(len(queries) + 1, dtype=np.int64)
    np.cumsum(np.bincount(b[keep], minlength=len(queries)), out=ptr[1:])
    return ptr, ids, vals


def run(name, est, side, queries, n_top, repeats, torch, kernel_time=False):
    h = est._h
    stream = torch.cuda.current_stream()
    h.set_stream(stream.cuda_stream)
    nq = len(queries)
    ptr, ids, vals = own_lists(est, queries)
    dq = torch.tensor(queries, dtype=torch.int32, device="cuda")
    d_ptr, d_ids, d_vals = (torch.from_numpy(x).cuda() for x in (ptr, ids, vals))
    out = {lab: (torch.empty((nq, n_top), dtype=torch.int32, device="cuda"),
                 torch.empty((nq, n_top), dtype=torch.float64, device="cuda")) for lab in ("by_id", "given")}

    def by_id():
        i, s = out["by_id"]
        h.recommend_device(side, dq.data_ptr(), nq, n_top, i.data_ptr(), s.data_ptr())

    def given():
        i, s = out["given"]
        h.recommend_given_device(side, d_ptr.data_ptr(), d_ids.data_ptr(), d_vals.data_ptr(), nq, n_top,
                                 i.data_ptr(), s.data_ptr())

    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    fns = {"by_id": by_id, "given": given}
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    times = {lab: [] for lab in fns}
    for _ in range(repeats):
        for lab, fn in fns.items():                      # alternated
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize()
            times[lab].append(a.elapsed_time(b))
    (ii, si), (gi, gs) = ((x.cpu().numpy(), y.cpu().numpy()) for x, y in (out["by_id"], out["given"]))
    ns, gn = np.isnan(si), np.isnan(gs)
    same = (np.array_equal(ii, gi) and np.array_equal(ns, gn)
            and np.array_equal(si[~ns].view(np.uint64), gs[~gn].view(np.uint64)))
    row = {"run": name, "side": side, "queries": nq, "n_top": n_top, "list_entries": int(ptr[-1]),
           "given_ms": round(float(np.median(times["given"])), 3),
           "by_id_ms": round(float(np.median(times["by_id"])), 3),
           "given_ms_all": [round(t, 3) for t in times["given"]], "by_id_ms_all": [round(t, 3) for t in times["by_id"]],
           "identical_lists": bool(same)}
    if side == "left":
        raters = np.bincount(est.Data.innerItems, minlength=est.Data.ItemCount)
        updates = float(raters[ids].sum())
        row["updates"] = updates
        if kernel_time:
            from torch.profiler import ProfilerActivity, profile

            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(repeats):
                    flush.zero_()
                    given()
                torch.cuda.synchronize()
            ks = [e for e in prof.key_averages() if "given_sims_kernel" in e.key]
            tot = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in ks)
            cnt = sum(e.count for e in ks)
            if cnt:
                k_ms = tot / cnt / 1e3
                row["given_sims_kernel_ms"] = round(k_ms, 3)
                row["given_sims_updates_per_s"] = updates / (k_ms * 1e-3)
    print(json.dumps(row), flush=True)
    h.set_stream(0, use_own=True)
    assert same, f"{name}: the given lists and the query ids list different targets"
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    import torch

    import bench
    import recommend_sys_b200 as rs

    if not torch.cuda.is_available():
        raise SystemExit("recommend_given_bench.py needs a CUDA device")
    print(json.dumps({"card": card()}), flush=True)
    if args.quick:
        train = rs.NewTrainSet(rs.core.synth_ratings(2000, 1500, 200_000, 0x5EED0042))
    else:
        train, _ = bench.make_data("ml20m_item_pearson_k40")
    est = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False, "k": 40}))
    est.Fit(train)
    est._h.synchronize()
    rng = np.random.RandomState(0x5EED)
    uniform = np.sort(rng.choice(train.UserCount, 1024, replace=False))
    run("ml20m_item_uniform", est, "right", uniform, 10, args.repeats, torch)
    est.Close()
    data = (rs.core.synth_ratings(800, 600, 60_000, 0x5EED0043) if args.quick
            else rs.core.synth_ratings(6040, 3706, 1_000_000, 0x5EED0044))
    train = rs.NewTrainSet(data)
    est = rs.NewKNN(rs.Parameters({"sim": rs.MSD, "userBased": True, "k": 40}))
    est.Fit(train)
    est._h.synchronize()
    run("ml1m_user_msd", est, "left", np.arange(train.UserCount), 10, args.repeats, torch, kernel_time=True)
    est.Close()
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
