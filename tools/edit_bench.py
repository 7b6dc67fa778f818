"""Removing or changing ratings of a fitted model (rs_knn_remove_device / rs_knn_change_device) against a Fit of the
edited ratings (rs_knn_fit_device), and where the edit stops paying.

For each workload and edit: handle A is fitted on all ratings (untimed) and then edited; handle B is fitted on the
edited ratings in the edited dataset order, under the same inner ids and counts.  Both timed calls run on the current
torch stream with CUDA events after a warm-up, alternated repeat by repeat, the L2 overwritten (a 512 MiB write) before
each, outside the timed window.  After the last repeat the two models are compared bit for bit: the whole matrix (in
row blocks), 200,000 predictions and the top-10 lists of 1,024 queries.
Workloads:
  ml20m_item   the ML-20M item shape (bench.py ml20m_item_pearson_k40), centered Pearson, k = 40, item-based;
  ml1m_user    the ML-1M user shape (synthetic, 6,040 x 3,706, 1 M ratings), MSD basic, k = 40, user-based.
Edits:
  remove_user       every rating of one user (the user with the median count);
  change_1024_users one rating of each of 1,024 users (their last one), r -> 6 - r;
  remove_1pct       a random 1 % of the ratings.
With --profile, one more edit per case runs under torch.profiler (CUDA activities) after the timed ones, and the
kernels that took the most device time are printed.
Usage: python tools/edit_bench.py [--repeats 5] [--quick] [--profile]"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from update_bench import card, last_per_group, same_models  # noqa: E402


def edits(train, rng):
    users = train.innerUsers
    counts = np.bincount(users, minlength=train.UserCount)
    median_user = int(np.argsort(counts, kind="stable")[len(counts) // 2])
    some = rng.choice(train.UserCount, min(1024, train.UserCount), replace=False)
    n = len(train.Ratings)
    return {"remove_user": ("remove", np.flatnonzero(users == median_user)),
            "change_1024_users": ("change", last_per_group(users, some)),
            "remove_1pct": ("remove", np.sort(rng.choice(n, n // 100, replace=False)))}


def run(name, train, kw, user_based, repeats, torch, rng, profile=False):
    import recommend_sys_b200 as rs

    left_all = (train.innerUsers if user_based else train.innerItems).astype(np.int32)
    right_all = (train.innerItems if user_based else train.innerUsers).astype(np.int32)
    n_left, n_right = (train.UserCount, train.ItemCount) if user_based else (train.ItemCount, train.UserCount)
    ratings = train.Ratings.astype(np.float64)
    stream = torch.cuda.current_stream()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    gm = float(np.mean(ratings))
    L, R, V = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (left_all, right_all, ratings))
    for ename, (kind, sel) in edits(train, rng).items():
        if kind == "remove":
            keep = np.ones(len(ratings), dtype=bool)
            keep[sel] = False
            el, er, ev = left_all[keep], right_all[keep], ratings[keep]
            new = None
        else:
            new = 6.0 - ratings[sel]
            el, er, ev = left_all, right_all, ratings.copy()
            ev[sel] = new
        EL, ER, EV = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (el, er, ev))
        DL, DR = (torch.from_numpy(np.ascontiguousarray(x[sel])).cuda() for x in (left_all, right_all))
        DV = torch.from_numpy(np.ascontiguousarray(new)).cuda() if new is not None else None
        nd, nnz = len(sel), len(ev)
        a, b = rs.core._Handle(**kw), rs.core._Handle(**kw)
        for h in (a, b):
            h.set_stream(stream.cuda_stream)

        def fit_all():
            a.fit_device(L.data_ptr(), R.data_ptr(), V.data_ptr(), len(ratings), n_left, n_right, gm)

        def edit():
            if DV is None:
                a.remove_device(DL.data_ptr(), DR.data_ptr(), nd, gm)
            else:
                a.change_device(DL.data_ptr(), DR.data_ptr(), DV.data_ptr(), nd, gm)

        def refit():
            b.fit_device(EL.data_ptr(), ER.data_ptr(), EV.data_ptr(), nnz, n_left, n_right, gm)

        fit_all(); edit(); refit()                            # warm-up
        torch.cuda.synchronize()
        times = {"edit": [], "refit": []}
        for _ in range(repeats):
            fit_all()
            for lab, fn in (("edit", edit), ("refit", refit)):
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

            fit_all()
            torch.cuda.synchronize()
            with prof_ctx(activities=[ProfilerActivity.CUDA]) as prof:
                edit()
                torch.cuda.synchronize()
            evs = sorted(prof.key_averages(), key=lambda e: -getattr(e, "device_time_total", 0.0))[:6]
            kernels = {e.key[:60]: round(getattr(e, "device_time_total", 0.0) / 1e3, 3) for e in evs}
        a.set_stream(0, use_own=True)
        b.set_stream(0, use_own=True)
        touched = len(np.unique(left_all[sel]))
        same = same_models(a, b, n_left, n_right, rng)
        row = {"run": name, "edit": ename, "pairs": nd, "touched_rows": touched, "n_left": n_left, "nnz": nnz,
               "edit_ms": round(float(np.median(times["edit"])), 3),
               "refit_ms": round(float(np.median(times["refit"])), 3),
               "edit_ms_all": [round(t, 3) for t in times["edit"]],
               "refit_ms_all": [round(t, 3) for t in times["refit"]], "identical": bool(same)}
        if kernels is not None:
            row["edit_kernels_ms"] = kernels
        print(json.dumps(row), flush=True)
        a.close()
        b.close()
        assert same, f"{name} {ename}: the edited model differs from the refit"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    ap.add_argument("--profile", action="store_true", help="device time of the edit's kernels, in a pass of its own")
    args = ap.parse_args()
    import torch

    import bench
    import recommend_sys_b200 as rs

    if not torch.cuda.is_available():
        raise SystemExit("edit_bench.py needs a CUDA device")
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
