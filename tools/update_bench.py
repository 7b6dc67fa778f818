"""Adding ratings to a fitted model (rs_knn_update_device) against a Fit of the union (rs_knn_fit_device), and where
the update stops paying.

For each workload and delta: D = every rating except the delta's, in dataset order, and the delta after it.  Handle A
is fitted on D (untimed) and then updated with the delta; handle B is fitted on D + delta.  Both timed calls run on the
current torch stream with CUDA events after a warm-up, alternated repeat by repeat, the L2 overwritten (a 512 MiB
write) before each, outside the timed window.  Both handles use the union's inner ids and counts, so D's Fit has empty
rows for ids only the delta rates.  After the last repeat the two models are compared bit for bit: the whole matrix
(in row blocks), 200,000 predictions and the top-10 lists of 1,024 queries.
Workloads:
  ml20m_item   the ML-20M item shape (bench.py ml20m_item_pearson_k40), centered Pearson, k = 40, item-based;
  ml1m_user    the ML-1M user shape (synthetic, 6,040 x 3,706, 1 M ratings), MSD basic, k = 40, user-based.
Deltas (one rating per row where a number of rows is named):
  one_user       one user's ratings (the user with the median count);
  1024_users     1,024 users' ratings;
  blockbusters   one rating of each of the 312 most-rated items;
  tenth_rows     one rating of each of a random tenth of the left rows (items, resp. users).
With --profile, one more update per delta runs under torch.profiler (CUDA activities) after the timed ones, and the
kernels that took the most device time are printed.
Usage: python tools/update_bench.py [--repeats 5] [--quick] [--profile]"""
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


def last_per_group(keys, groups):
    """Positions of the last rating (in dataset order) of every key in `groups`."""
    pos = np.full(int(keys.max()) + 1, -1, dtype=np.int64)
    pos[keys] = np.arange(len(keys))              # the last write wins: the last position
    return np.sort(pos[groups])


def deltas(train, user_based, rng):
    users, items = train.innerUsers, train.innerItems
    counts = np.bincount(users, minlength=train.UserCount)
    median_user = int(np.argsort(counts, kind="stable")[len(counts) // 2])
    some = rng.choice(train.UserCount, min(1024, train.UserCount), replace=False)
    pop = np.argsort(-np.bincount(items, minlength=train.ItemCount), kind="stable")[:312]
    left = users if user_based else items
    n_left = train.UserCount if user_based else train.ItemCount
    tenth = rng.choice(n_left, n_left // 10, replace=False)
    return {"one_user": np.flatnonzero(users == median_user),
            "1024_users": np.flatnonzero(np.isin(users, some)),
            "blockbusters": last_per_group(items, pop),
            "tenth_rows": last_per_group(left, tenth)}


def same_models(a, b, n_left, n_right, rng):
    block = 1024
    for r0 in range(0, n_left, block):
        nr = min(block, n_left - r0)
        x, y = a.sims_rows(r0, nr), b.sims_rows(r0, nr)
        if not (np.array_equal(np.isnan(x), np.isnan(y)) and np.array_equal(np.nan_to_num(x).view(np.uint64),
                                                                           np.nan_to_num(y).view(np.uint64))):
            return False
    left = rng.randint(0, n_left, 200_000).astype(np.int32)
    right = rng.randint(0, n_right, 200_000).astype(np.int32)
    pa, pb = a.predict_batch(left, right), b.predict_batch(left, right)
    if not np.array_equal(np.nan_to_num(pa, nan=7e300).view(np.uint64), np.nan_to_num(pb, nan=7e300).view(np.uint64)):
        return False
    q = rng.choice(n_left, min(1024, n_left), replace=False)
    ia, sa = a.recommend("left", q, 10)
    ib, sb = b.recommend("left", q, 10)
    return np.array_equal(ia, ib) and np.array_equal(np.nan_to_num(sa, nan=7e300).view(np.uint64),
                                                     np.nan_to_num(sb, nan=7e300).view(np.uint64))


def run(name, train, kw, user_based, repeats, torch, rng, profile=False):
    import recommend_sys_b200 as rs

    left_all = train.innerUsers if user_based else train.innerItems
    right_all = train.innerItems if user_based else train.innerUsers
    n_left, n_right = (train.UserCount, train.ItemCount) if user_based else (train.ItemCount, train.UserCount)
    stream = torch.cuda.current_stream()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    for dname, sel in deltas(train, user_based, rng).items():
        rest = np.ones(len(train.Ratings), dtype=bool)
        rest[sel] = False
        order = np.concatenate([np.flatnonzero(rest), sel])
        gm = float(np.mean(train.Ratings))
        L, R, V = (torch.from_numpy(np.ascontiguousarray(x[order])).cuda() for x in (left_all.astype(np.int32),
                                                                              right_all.astype(np.int32),
                                                                              train.Ratings.astype(np.float64)))
        nd, nnz = len(sel), len(order)
        m = nnz - nd
        a, b = rs.core._Handle(**kw), rs.core._Handle(**kw)
        for h in (a, b):
            h.set_stream(stream.cuda_stream)

        def fit_d():
            a.fit_device(L.data_ptr(), R.data_ptr(), V.data_ptr(), m, n_left, n_right, gm)

        def update():
            a.update_device(L[m:].data_ptr(), R[m:].data_ptr(), V[m:].data_ptr(), nd, n_left, n_right, gm)

        def refit():
            b.fit_device(L.data_ptr(), R.data_ptr(), V.data_ptr(), nnz, n_left, n_right, gm)

        fit_d(); update(); refit()                            # warm-up
        torch.cuda.synchronize()
        times = {"update": [], "refit": []}
        for _ in range(repeats):
            fit_d()
            for lab, fn in (("update", update), ("refit", refit)):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                torch.cuda.synchronize()
                times[lab].append(e0.elapsed_time(e1))
        kernels = None
        if profile:
            from torch.profiler import ProfilerActivity, profile as prof_ctx

            fit_d()
            torch.cuda.synchronize()
            with prof_ctx(activities=[ProfilerActivity.CUDA]) as prof:
                update()
                torch.cuda.synchronize()
            ev = sorted(prof.key_averages(), key=lambda e: -getattr(e, "device_time_total", 0.0))[:6]
            kernels = {e.key[:60]: round(getattr(e, "device_time_total", 0.0) / 1e3, 3) for e in ev}
        a.set_stream(0, use_own=True)
        b.set_stream(0, use_own=True)
        touched = len(np.unique(left_all[sel]))
        same = same_models(a, b, n_left, n_right, rng)
        row = {"run": name, "delta": dname, "ratings": nd, "touched_rows": touched, "n_left": n_left, "nnz": nnz,
               "update_ms": round(float(np.median(times["update"])), 3),
               "refit_ms": round(float(np.median(times["refit"])), 3),
               "update_ms_all": [round(t, 3) for t in times["update"]],
               "refit_ms_all": [round(t, 3) for t in times["refit"]], "identical": bool(same)}
        if kernels is not None:
            row["update_kernels_ms"] = kernels
        print(json.dumps(row), flush=True)
        a.close()
        b.close()
        assert same, f"{name} {dname}: the updated model differs from the refit"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    ap.add_argument("--profile", action="store_true", help="device time of the update's kernels, in a pass of its own")
    args = ap.parse_args()
    import torch

    import bench
    import recommend_sys_b200 as rs

    if not torch.cuda.is_available():
        raise SystemExit("update_bench.py needs a CUDA device")
    print(json.dumps({"card": card()}), flush=True)
    rng = np.random.RandomState(0x5EED)
    if args.quick:
        train = rs.NewTrainSet(rs.core.synth_ratings(2000, 1500, 200_000, 0x5EED0042))
    else:
        train, _ = bench.make_data("ml20m_item_pearson_k40")
    run("ml20m_item", train, dict(sim="pearson", knn_type="centered", k=40), False, args.repeats, torch, rng,
        args.profile)
    data = (rs.core.synth_ratings(800, 600, 60_000, 0x5EED0043) if args.quick
            else rs.core.synth_ratings(6040, 3706, 1_000_000, 0x5EED0044))
    run("ml1m_user", rs.NewTrainSet(data), dict(sim="msd", knn_type="basic", k=40), True, args.repeats, torch, rng,
        args.profile)
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
