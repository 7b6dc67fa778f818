"""Adding ratings to cyclic row shards (rs_knn_update_sharded_device): the update time of each shard against R = 1, a
full handle updated by rs_knn_update_device.

Every shard of R = 2, 4 and 8 shards of one model lives on the current GPU and runs one after another, so each
shard's time is the time it would take on a GPU of its own (the update exchanges no data).  For each workload and
delta: D = every rating except the delta's, in dataset order, and the delta after it (as tools/update_bench.py).  Per
repeat the shards are fitted on D and mirrored (untimed), then each shard's update is timed with CUDA events on the
current torch stream, the L2 overwritten (a 512 MiB write) before each, outside the timed window.  In a pass of its
own, each shard's update runs under torch.profiler and the device time of given_sims_kernel (both variants) is
summed.  After the last repeat each shard's rows are compared bit for bit with the same shard of a cyclic Fit of the
union (R = 1: the full handle against a Fit of the union).
Workloads (tools/update_bench.py):
  ml20m_item   the ML-20M item shape (bench.py ml20m_item_pearson_k40), centered Pearson, k = 40, item-based;
  ml1m_user    the ML-1M user shape (synthetic, 6,040 x 3,706, 1 M ratings), MSD basic, k = 40, user-based.
Deltas: one_user (the user with the median count), 1024_users, tenth_rows (one rating of each of a random tenth of
the left rows).
Expected, from the algorithm (not a measurement): a shard does about 2 T N / R of the T N similarity work of R = 1.
Usage: python tools/update_shard_bench.py [--repeats 3] [--shards 2,4,8] [--quick]"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from update_bench import card, deltas  # noqa: E402


def same_rows(a, b, rows, n_left):
    """The rows `rows` (global ids, in storage order) of two handles, bit for bit, read a 32-row block at a time."""
    for blk in np.split(rows, np.flatnonzero(np.diff(rows) != 1) + 1):
        for r0 in range(0, len(blk), 1024):
            part = blk[r0:r0 + 1024]
            if len(part) == 0:
                continue
            x, y = a.sims_rows(int(part[0]), len(part)), b.sims_rows(int(part[0]), len(part))
            if not (np.array_equal(np.isnan(x), np.isnan(y)) and
                    np.array_equal(np.nan_to_num(x).view(np.uint64), np.nan_to_num(y).view(np.uint64))):
                return False
    return True


def given_ms(prof):
    return sum(getattr(e, "device_time_total", 0.0) for e in prof.key_averages() if "given_sims_kernel" in e.key) / 1e3


def run(name, train, kw, user_based, counts, repeats, torch, rng):
    import recommend_sys_b200 as rs
    from torch.profiler import ProfilerActivity, profile

    left_all = train.innerUsers if user_based else train.innerItems
    right_all = train.innerItems if user_based else train.innerUsers
    n_left, n_right = (train.UserCount, train.ItemCount) if user_based else (train.ItemCount, train.UserCount)
    stream = torch.cuda.current_stream()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    all_deltas = deltas(train, user_based, rng)
    for dname in ("one_user", "1024_users", "tenth_rows"):
        sel = all_deltas[dname]
        rest = np.ones(len(train.Ratings), dtype=bool)
        rest[sel] = False
        order = np.concatenate([np.flatnonzero(rest), sel])
        gm = float(np.mean(train.Ratings))
        L, Rr, V = (torch.from_numpy(np.ascontiguousarray(x[order])).cuda() for x in (left_all.astype(np.int32),
                                                                               right_all.astype(np.int32),
                                                                               train.Ratings.astype(np.float64)))
        nd, nnz = len(sel), len(order)
        m = nnz - nd
        touched = len(np.unique(left_all[sel]))

        def fit(hs, n):
            for h in hs:
                h.fit_device(L.data_ptr(), Rr.data_ptr(), V.data_ptr(), n, n_left, n_right, gm)
            if len(hs) > 1:
                torch.cuda.synchronize()
                for h in hs:
                    h.peer_import_local(hs)
                    h.mirror()
            torch.cuda.synchronize()

        def update(h, sharded):
            call = h.update_sharded_device if sharded else h.update_device
            call(L[m:].data_ptr(), Rr[m:].data_ptr(), V[m:].data_ptr(), nd, n_left, n_right, gm)

        for count in [1] + counts:
            shard_kw = [dict(kw)] if count == 1 else [dict(kw, shard_count=count, shard_index=q) for q in range(count)]
            hs = [rs.core._Handle(**k) for k in shard_kw]
            for h in hs:
                h.set_stream(stream.cuda_stream)
            times = [[] for _ in hs]
            for rep in range(repeats + 1):                  # the first pass warms up
                fit(hs, m)
                for q, h in enumerate(hs):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    update(h, count > 1)
                    e1.record(stream)
                    torch.cuda.synchronize()
                    if rep:
                        times[q].append(e0.elapsed_time(e1))
            fit(hs, m)
            kern = []
            for h in hs:
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    update(h, count > 1)
                    torch.cuda.synchronize()
                kern.append(given_ms(prof))
            ref = [rs.core._Handle(**k) for k in shard_kw]
            for h in ref:
                h.set_stream(stream.cuda_stream)
            fit(ref, nnz)
            for q, (h, g) in enumerate(zip(hs, ref)):
                rows = rs.core.cyclic_rows(n_left, count, q) if count > 1 else np.arange(n_left)
                same = same_rows(h, g, rows, n_left)
                print(json.dumps({"run": name, "delta": dname, "ratings": nd, "touched_rows": touched,
                                  "n_left": n_left, "shards": count, "shard": q, "rows": int(len(rows)),
                                  "update_ms": round(float(np.median(times[q])), 3),
                                  "update_ms_all": [round(t, 3) for t in times[q]],
                                  "given_sims_kernel_ms": round(kern[q], 3), "identical": bool(same)}), flush=True)
                assert same, f"{name} {dname} R={count} shard {q}: the updated rows differ from the Fit of the union"
            for h in hs + ref:
                h.set_stream(0, use_own=True)
                h.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--shards", default="2,4,8")
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    import torch

    import bench
    import recommend_sys_b200 as rs

    if not torch.cuda.is_available():
        raise SystemExit("update_shard_bench.py needs a CUDA device")
    counts = [int(c) for c in args.shards.split(",")]
    print(json.dumps({"card": card()}), flush=True)
    rng = np.random.RandomState(0x5EED)
    if args.quick:
        train = rs.NewTrainSet(rs.core.synth_ratings(2000, 1500, 200_000, 0x5EED0042))
    else:
        train, _ = bench.make_data("ml20m_item_pearson_k40")
    run("ml20m_item", train, dict(sim="pearson", knn_type="centered", k=40), False, counts, args.repeats, torch, rng)
    data = (rs.core.synth_ratings(800, 600, 60_000, 0x5EED0043) if args.quick
            else rs.core.synth_ratings(6040, 3706, 1_000_000, 0x5EED0044))
    run("ml1m_user", rs.NewTrainSet(data), dict(sim="msd", knn_type="basic", k=40), True, counts, args.repeats, torch,
        rng)
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
