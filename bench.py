#!/usr/bin/env python
"""bench.py — the KNN hot path (Fit = all-pairs similarity, then full test-set Predict) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU algorithm

One "step" = one pass of the hot path over one synthetic rating matrix.  The default workload is the
north-star target of BASELINE.json: KNNWithMeans, item-based Pearson (exact mode: bit-identical to the
reference), k = 40, MovieLens-20M shape (138,493 x 26,744 with 20,000,000 training ratings; the test set
is a further 4,000,000 held-out pairs of the same generator):
    Fit(train)    -> dense N x N float64 similarity matrix resident in HBM (N = 26,744 items, 5.7 GB)
    Predict(test) -> 4,000,000 predictions
metric = similarity pairs/s = N(N-1)/2 unordered left-row pairs / step time (Fit + Predict);
predictions/s over the same step is reported beside it.  `value` is timed with CUDA events with
every input already resident in HBM; `e2e` is the same step through the public API with HOST
buffers (pinned), host<->device copies inside the timed region.  Other BASELINE.json configs are
selectable with --workload (configs[1] = ml1m_item_pearson_k40).

--steps K times exactly K steps of each kind (device and e2e).  --dump-outputs DIR writes what the last
timed device step computed (predictions, similarity rows, neighbour lists; seeded samples where larger
than the 64 MB budget; NaN and infinities as a separate mask, see dump_outputs) as .npy files of finite
numbers: the inputs are generated from fixed seeds, so two builds run with the same arguments can be
compared output for output.

N > 1 (torchrun, one rank per GPU): STRONG scaling of that ONE matrix.  The exact sparse path runs as
cyclic row shards — every pair is computed once across the ranks, the other triangle of a rank's rows is
pulled from the peers' matrices over NVLink, each rank predicts the test pairs whose left row it owns and
the predictions are all-gathered (NCCL) inside the timed region.  Tensor-path workloads use contiguous
row shards, top-k-only workloads symmetric slabs.  `--folds` gives a fold per GPU instead (weak).

The reference arm times the CPU restatement of the Go algorithm (oracle/, the reference itself
is Go and no Go toolchain exists in the image) on the box's host cores: Fit with nJobs = all
cores exactly as core/knn.go:192-216, Predict as the reference's serial loop (core/data.go:98-105).
Under torchrun rank 0 alone runs it, on the full workload whatever N is.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (users, items, train nnz, test nnz, sim, knn_type, user_based, k)
    "ml1m_item_pearson_k40": (6040, 3706, 1_000_000, 200_000, "pearson", "centered", False, 40),
    "ml100k_user_cosine_k40": (943, 1682, 80_000, 20_000, "cosine", "basic", True, 40),
    "ml1m_item_cosine_k40": (6040, 3706, 1_000_000, 200_000, "cosine", "basic", False, 40),
    "ml1m_item_msd_k40": (6040, 3706, 1_000_000, 200_000, "msd", "basic", False, 40),
    "ml20m_item_cosine_k40": (138_493, 26_744, 20_000_000, 4_000_000, "cosine", "basic", False, 40),
    "ml20m_item_msd_k40": (138_493, 26_744, 20_000_000, 4_000_000, "msd", "basic", False, 40),
    "ml20m_item_pearson_k40": (138_493, 26_744, 20_000_000, 4_000_000, "pearson", "centered", False, 40),
    "ml20m_item_pearson_baseline_k40": (138_493, 26_744, 20_000_000, 4_000_000, "pearson_baseline", "baseline", False, 40),
    "ml20m_user_msd_k100": (138_493, 26_744, 20_000_000, 0, "msd", "basic", True, 100),
    # SURVEY.md §8 f-2: Slope One (core/slope_one.go) — item x item deviation matrix + full test-set Predict
    "ml1m_slope_one": (6040, 3706, 1_000_000, 200_000, "slope_one", "basic", False, 40),   # k unused
    "ml20m_slope_one": (138_493, 26_744, 20_000_000, 4_000_000, "slope_one", "basic", False, 40),
    "netflix_item_cosine_k50": (480_189, 17_770, 100_000_000, 20_000_000, "cosine", "basic", False, 50),
}
DEFAULT_WORKLOAD = "ml20m_item_pearson_k40"
SEED = 0x5EED0000 + 1  # config index 1 (SURVEY.md §8d)


def make_data(workload, fold=0):
    import recommend_sys_b200 as rs

    users, items, nnz, n_test, *_ = WORKLOADS[workload]
    d = rs.core.synth_ratings(users, items, nnz + n_test, SEED + 1000 * fold)
    test = d.SubSet(np.arange(0, n_test))
    train = rs.NewTrainSet(d.SubSet(np.arange(n_test, d.Length())))
    return train, test


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [x for x in sm if x >= 0.5 * max(sm)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return float(j["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def cpu_reference_step(ob, ots, test, sim, knn_type, user_based, k, cores, rows=None, n_pred=None):
    """One step of the reference's CPU algorithm (restated in oracle/): returns (seconds_fit,
    seconds_predict, rows_fitted, n_predicted)."""
    if sim == "slope_one":      # core/slope_one.go: Fit on all cores, serial Predict loop (core/data.go:98-105)
        n_items = ots.item_count
        # a slab is taken at the END of the matrix: row i meets its i predecessors (core/slope_one.go:72),
        # so the last m rows do ~m*n pair merges — the same scaling rule as the KNN slabs
        srows = None if rows is None else (n_items - (rows[1] - rows[0]), n_items)
        t0 = time.perf_counter()
        so = ob.SlopeOne().fit(ots, n_jobs=cores, rows=srows)
        t1 = time.perf_counter()
        u, i = test.Users, test.Items
        if n_pred is not None:
            u, i = u[:n_pred], i[:n_pred]
        t2 = time.perf_counter()
        so.predict_batch(u, i)
        t3 = time.perf_counter()
        return t1 - t0, t3 - t2, (n_items if rows is None else rows[1] - rows[0]), len(u)
    # config 3 (PearsonBaseline + KNNBaseline) uses ALS baselines on both arms (BASELINE.json configs[2])
    knn = ob.KNN(sim=sim, knn_type=knn_type, user_based=user_based, k=k, n_jobs=cores, tie_policy="go",
                 baseline="als" if sim == "pearson_baseline" else "sgd")
    t0 = time.perf_counter()
    knn.fit(ots, rows=rows)
    t1 = time.perf_counter()
    u, i = test.Users, test.Items
    if rows is not None:
        inner = (ots_inner(ots, user_based))
        left_of_test = inner(u if user_based else i)
        sel = np.where((left_of_test >= rows[0]) & (left_of_test < rows[1]))[0]
        u, i = u[sel], i[sel]
    if n_pred is not None:
        u, i = u[:n_pred], i[:n_pred]
    t2 = time.perf_counter()
    knn.predict_batch(u, i, n_threads=1)  # the reference's loop is serial (core/data.go:98-105)
    t3 = time.perf_counter()
    return t1 - t0, t3 - t2, (knn.n if rows is None else rows[1] - rows[0]), len(u)


def ots_inner(ots, user_based):
    from oracle import binding as ob

    L = ob.lib()
    conv = L.or_trainset_convert_user if user_based else L.or_trainset_convert_item
    return lambda raw: np.array([conv(ots.h, int(x)) for x in raw], dtype=np.int64)


def representative_slab(left_inner, n, rows):
    """A contiguous slab of `rows` left rows whose mean length is closest to the mean over all rows
    (deterministic).  A CPU merge-join Fit pays about N*len(i) + nnz steps for row i, so a slab of the
    longest rows (the low ids) would overstate the cost of the whole matrix by an order of magnitude."""
    deg = np.bincount(left_inner, minlength=n).astype(np.float64)
    if rows >= n:
        return 0, n
    c = np.concatenate([[0.0], np.cumsum(deg)])
    means = (c[rows:] - c[:-rows]) / rows
    i0 = int(np.argmin(np.abs(means - deg.mean())))
    return i0, i0 + rows


def cpu_sample_rows(n, nnz, budget_merge_steps):
    """Rows of a Fit slab that cost about `budget_merge_steps` two-pointer steps (2*nnz per row on average)."""
    rows = int(budget_merge_steps / (2.0 * nnz))
    if rows >= n:
        return n
    # at least 24 rows per host thread: the reference splits the rows statically over nJobs threads
    # (core/knn.go:192-199) and a slab of a few rows per thread measures the imbalance, not the algorithm
    floor = min(n, 24 * (os.cpu_count() or 1))
    return max(floor, rows // 64 * 64)


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (restated), on rank 0,
    on the FULL workload whatever N is (the other ranks exit without work)."""
    if rank != 0:
        return
    from oracle import binding as ob

    users, items, nnz, n_test, sim, knn_type, user_based, k = WORKLOADS[args.workload]
    train, test = make_data(args.workload)
    ots = ob.TrainSet(train.Users, train.Items, train.Ratings)
    cores = os.cpu_count() or 1
    n = train.UserCount if user_based else train.ItemCount
    left_inner = train.innerUsers if user_based else train.innerItems
    pairs_full = n * (n - 1) / 2
    total_steps = args.steps + args.warmup
    # a bounded, DETERMINISTIC sample: the slab size follows from the workload and K + W only
    # (about 150 s of 16-thread merge-join work over the whole run, ~6e8 steps/s), never from a timing probe
    nrows = cpu_sample_rows(n, train.Length(), 9e10 / max(1, total_steps))
    if nrows >= n:
        rows, n_pred, sample = None, None, f"full workload: Fit all {n} rows + {test.Length()} serial predictions"
        if test.Length() > 200_000:
            n_pred = 200_000 // max(1, total_steps) * 4
            sample = f"full Fit of all {n} rows + first {n_pred} test pairs predicted serially (scaled)"
    else:
        rows = representative_slab(left_inner, n, nrows)
        n_pred = max(1000, 40_000 // max(1, total_steps) * 4)
        sample = (f"Fit slab of rows [{rows[0]},{rows[1]}) of {n} (mean row length closest to the matrix mean) x all {n} "
                  f"columns, scaled x{n / nrows:.1f}/2 + first {n_pred} of the slab's test pairs predicted serially, scaled")
    times = []
    for s in range(total_steps):
        tf, tp, rows_done, npred = cpu_reference_step(ob, ots, test, sim, knn_type, user_based, k, cores, rows=rows,
                                                      n_pred=n_pred)
        if s >= args.warmup:
            times.append((tf, tp, rows_done, npred))
    tf = sum(t[0] for t in times) / len(times)
    tp = sum(t[1] for t in times) / len(times)
    rows_done, npred = times[0][2], times[0][3]
    # the slab computes rows_done x (n-1) ordered pairs; a full Fit computes every unordered
    # pair once (core/knn.go:203 skips filled cells), i.e. n/rows_done/2 slabs' worth
    fit_s = tf if rows is None else tf * (n / rows_done) * 0.5
    pred_s = (tp / max(1, npred)) * test.Length()
    step_s = fit_s + pred_s
    value = pairs_full / step_s
    line = {
        "impl": "reference", "metric": "similarity_pairs_per_sec", "value": value, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.gpus > 1 and not args.folds else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "predictions_per_sec": test.Length() / step_s,
        "fit_ms": fit_s * 1e3, "predict_ms": pred_s * 1e3,
        "config": {"workload": args.workload, "shape": f"{users}x{items}", "train_ratings": train.Length(),
                   "test_pairs": test.Length(), "sim": sim, "knn_type": knn_type, "user_based": user_based, "k": k,
                   "tie_policy": "go (pdqsort port)"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def pinned_like(a):
    """A numpy view over page-locked host memory holding a copy of `a`."""
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    _KEEP.append(t)
    return t.numpy()


_KEEP = []

# --dump-outputs: all files together stay under 64 MB (DUMP_BYTES leaves room for the .npy headers); larger
# outputs are sampled, with the same seeded rows or entries on every run, so that two builds can be compared
# array by array.  Every file holds finite numbers only: a NaN or infinite value (an unset similarity, a
# prediction without neighbours) is written as 0.0 in <name>.npy and its kind in <name>_nonfinite.npy
# (float32, same shape: 0 finite, 1 NaN, 2 +inf, 3 -inf), so the budgets count 8 + 4 bytes per value.
DUMP_BYTES = 63_000_000
DUMP_PRED_BYTES = 48_000_000      # the predictions' share: all 4 M of the MovieLens-20M test set
DUMP_SEED = 0


def _dump_sample(n, cap):
    """Positions 0..n-1, or a sorted seeded sample of `cap` of them."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, cap, replace=False))


def dump_outputs(out_dir, h, d_pred, lists, n_pred, store_matrix):
    """Writes what one step of the timed path returned as out_dir/<name>.npy, float64 throughout (ids too):
    predictions.npy, in test-set order (predictions_index.npy: which test pairs, when sampled);
    matrix.npy, rows matrix_rows.npy of the similarity matrix the handle holds; topk_index.npy (-1: no
    neighbour) and topk_sims.npy, rows topk_rows.npy of the neighbour lists; <name>_nonfinite.npy beside
    an output that had NaN or infinite values."""
    import torch

    out_dir.mkdir(parents=True, exist_ok=True)

    def save(name, a):
        a = np.asarray(a, dtype=np.float64)
        bad = ~np.isfinite(a)
        if bad.any():
            kind = np.where(np.isnan(a), 1, np.where(a > 0, 2, 3)) * bad
            np.save(out_dir / f"{name}_nonfinite.npy", kind.astype(np.float32))
            a = np.where(bad, 0.0, a)
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a))

    left = DUMP_BYTES
    if d_pred is not None:
        full = n_pred * 12 <= DUMP_PRED_BYTES
        per = 12 if full else 20                                   # value + kind (+ index when sampled)
        sel = _dump_sample(n_pred, DUMP_PRED_BYTES // per)
        save("predictions", d_pred[torch.from_numpy(sel).to(d_pred.device)].cpu().numpy())
        if not full:
            save("predictions_index", sel)
        left -= len(sel) * per
    share = left // max(1, int(store_matrix) + int(lists is not None))
    if store_matrix:
        owned = h.owned_rows()
        rows = owned[_dump_sample(len(owned), share // (12 * h.n_left + 8))]
        save("matrix", np.concatenate([h.sims_rows(int(r), 1) for r in rows]))
        save("matrix_rows", rows)
    if lists is not None:
        idx, sims = lists
        rows = _dump_sample(idx.shape[0], share // (20 * idx.shape[1] + 8))
        d_rows = torch.from_numpy(rows).to(idx.device)
        save("topk_index", idx[d_rows].cpu().numpy())
        save("topk_sims", sims[d_rows].cpu().numpy())
        save("topk_rows", rows)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import recommend_sys_b200 as rs
    from recommend_sys_b200.shard import (ShardedKNN, allgather_partial_topk, allgather_predictions, allgather_topk,
                                          attach_peers_and_mirror, route_pairs, shard_rows, union_topk_device)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this framework has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    users, items, nnz, n_test, sim, knn_type, user_based, k = WORKLOADS[args.workload]
    # How N > 1 GPUs share ONE matrix (strong scaling; --folds restores a fold per GPU, weak):
    #   sym    top-k-only workloads (config 4: no test set, the N x N matrix would not fit): SYMMETRIC SLABS,
    #          every pair once, slabs dealt in snake order, all-gather + union of partial neighbour lists
    #   cyc    exact sparse path (Pearson exact, PearsonBaseline, --sim-path stream): CYCLIC ROW SHARDS, every
    #          pair once, the other triangle pulled from the peers over NVLink, test pairs routed to the owner
    #          of their left row, predictions all-gathered
    #   shard  tensor path: contiguous 128-aligned row shards (full rows), all-gather of lists and predictions
    sym = n_test == 0
    multi = world > 1 and not args.folds
    stream_exact = (sim in ("pearson", "pearson_baseline") and args.pearson_mode == "exact") or args.sim_path == "stream"
    cyc = multi and not sym and stream_exact and not args.shard_rows
    shard = multi and not sym and not cyc
    train, test = make_data(args.workload, fold=rank if (world > 1 and args.folds) else 0)
    n_left = train.UserCount if user_based else train.ItemCount
    n_right = train.ItemCount if user_based else train.UserCount
    left = train.innerUsers if user_based else train.innerItems
    right = train.innerItems if user_based else train.innerUsers
    t_left_raw = test.Users if user_based else test.Items
    t_right_raw = test.Items if user_based else test.Users
    t_left = (train.convert_users if user_based else train.convert_items)(t_left_raw)
    t_right = (train.convert_items if user_based else train.convert_users)(t_right_raw)
    rb, re = shard_rows(n_left, world, rank) if shard else (0, 0)
    counts = None
    mine = None
    if shard and n_test:
        mine = (t_left >= rb) & (t_left < re)
    if cyc:
        # every rank gets the full test set, answers the pairs whose left row it owns (+0.0 elsewhere) and an
        # int64 SUM all-reduce of the bit patterns assembles the predictions: no routing, no re-ordering
        own_cyc = route_pairs(t_left, world) == rank
        n_mine_cyc = int(own_cyc.sum())
    if mine is not None:
        t_left, t_right = t_left[mine], t_right[mine]
    n_pred = len(t_left)

    stream = torch.cuda.Stream(device=dev)   # a dedicated (non-default) stream for the whole bench
    torch.cuda.set_stream(stream)
    h = rs.core._Handle(sim=sim, knn_type=knn_type, k=k, device=local_rank, row_begin=rb, row_end=re,
                        store="topk" if sym else "matrix", topk=k,
                        shard_count=world if ((sym and not args.folds) or cyc) else (1 if sym else 0),
                        shard_index=rank if ((sym and not args.folds) or cyc) else 0,
                        pearson_mode=args.pearson_mode, sim_path=args.sim_path)
    h.set_stream(stream.cuda_stream)

    d_left = torch.from_numpy(left).to(dev)
    d_right = torch.from_numpy(right).to(dev)
    d_rating = torch.from_numpy(train.Ratings).to(dev)
    # KNNBaseline / PearsonBaseline take the bias vectors of the (host, sequential SGD) baseline
    # model as inputs (core/knn.go:179-187, core/base.go:135-163); they are computed once here and
    # are device-resident inputs of the timed step, like the ratings
    d_lb = d_rb = None
    global_bias = 0.0
    if knn_type == "baseline" or sim == "pearson_baseline":
        bl = rs.NewBaseLine(rs.Parameters({"baseline": "als" if sim == "pearson_baseline" else "sgd",
                                           "device": local_rank}))
        bl.Fit(train)
        lb, rbias = (bl.userBias, bl.itemBias) if user_based else (bl.itemBias, bl.userBias)
        global_bias = float(bl.globalBias)
        d_lb = torch.from_numpy(np.ascontiguousarray(lb, dtype=np.float64)).to(dev)
        if sim == "pearson_baseline":
            d_rb = torch.from_numpy(np.ascontiguousarray(rbias, dtype=np.float64)).to(dev)
    d_tl = torch.from_numpy(t_left).to(dev) if n_pred else None
    d_tr = torch.from_numpy(t_right).to(dev) if n_pred else None
    d_out = torch.empty(max(1, n_pred), dtype=torch.float64, device=dev)
    rows_local = (re - rb) if shard else n_left
    d_tk_i = torch.empty((rows_local, k), dtype=torch.int32, device=dev) if (shard or sym) else None
    d_tk_s = torch.empty((rows_local, k), dtype=torch.float64, device=dev) if (shard or sym) else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_device():
        """One step; returns what a caller of the path receives besides the similarity matrix that stays in
        `h`: (predictions, neighbour lists), None where the workload has none."""
        h.fit_device(d_left.data_ptr(), d_right.data_ptr(), d_rating.data_ptr(), len(left), n_left, n_right,
                     train.GlobalMean, d_lb.data_ptr() if d_lb is not None else 0,
                     d_rb.data_ptr() if d_rb is not None else 0, global_bias)
        if cyc:
            attach_peers_and_mirror(h)          # the exchange step: other triangle over NVLink
        if cyc:
            h.predict_batch_sharded_device(d_tl.data_ptr(), d_tr.data_ptr(), n_pred, d_out.data_ptr())
            dist.all_reduce(d_out.view(torch.int64), op=dist.ReduceOp.SUM)
            return d_out, None
        if n_pred:
            h.predict_batch_device(d_tl.data_ptr(), d_tr.data_ptr(), n_pred, d_out.data_ptr())
        lists = None
        if shard:
            h.topk_device(k, d_tk_i.data_ptr(), d_tk_s.data_ptr())
            lists = allgather_topk(d_tk_i, d_tk_s, n_left, k)
        if sym:
            h.topk_device(k, d_tk_i.data_ptr(), d_tk_s.data_ptr())
            lists = union_topk_device(*allgather_partial_topk(d_tk_i, d_tk_s)) if multi else (d_tk_i, d_tk_s)
        return (d_out if n_pred else None), lists

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    clocks.start()          # started before the warm-up: NVML start-up must not overlap the timed region
    for _ in range(args.warmup):
        step_device()
        flush.fill_(1)
    barrier()
    h.profile_reset()
    clocks.rows.clear()     # keep only the samples taken during the timed region
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for s in range(args.steps):
        ev[s][0].record(stream)
        result = step_device()
        ev[s][1].record(stream)
        flush.fill_(s & 0xff)  # L2 flush between timed iterations (outside the event pairs)
    barrier()
    clock_info = clocks.stop()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    prof = h.profile()
    if args.dump_outputs and rank == 0:     # before the e2e steps, which reuse the neighbour-list buffers
        dump_outputs(Path(args.dump_outputs), h, *result, n_pred, store_matrix=not sym)

    # ---- e2e: public API, host (pinned) buffers in, host predictions out ----
    train.innerUsers = pinned_like(train.innerUsers)
    train.innerItems = pinned_like(train.innerItems)
    train.Ratings = pinned_like(train.Ratings)
    ctor = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore,
            "baseline": rs.NewKNNBaseLine}[knn_type]
    if sim == "slope_one":
        ctor = rs.NewSlopeOne
    sim_obj = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson, "pearson_baseline": rs.PearsonBaseline,
               "slope_one": None}[sim]
    params = {"sim": sim_obj, "userBased": user_based, "k": k, "device": local_rank,
              "pearsonMode": args.pearson_mode, "simPath": args.sim_path}
    if sim == "pearson_baseline":
        params["baseline"] = "als"      # device ALS baselines inside the timed e2e Fit
    if shard:
        params.update({"rowBegin": rb, "rowEnd": re})
    if sym:
        params.update({"store": "topk", "topk": k, "shardCount": world if multi else 1, "shardIndex": rank if multi else 0})
    e2e_test = test
    if shard and n_test:
        e2e_test = test.SubSet(np.where(mine)[0])

    def step_e2e():
        if cyc:     # Fit + Predict of the ONE matrix on all ranks through the sharded estimator
            est = ShardedKNN(ctor(rs.Parameters(params)))
            est.Fit(train)
            out = est.PredictBatch(test.Users, test.Items)
            est.Close()
            return out
        est = ctor(rs.Parameters(params))
        est.Fit(train)
        out = e2e_test.Predict(est) if n_test else None
        if sym:     # the result of a top-k-only Fit is the neighbour lists: united across ranks, read to the host
            est._h.topk_device(k, d_tk_i.data_ptr(), d_tk_s.data_ptr())
            est._h.synchronize()     # the estimator works on its own stream; the union below on torch's
            li, ls = (union_topk_device(*allgather_partial_topk(d_tk_i, d_tk_s)) if multi else (d_tk_i, d_tk_s))
            out = (li.cpu(), ls.cpu())
        est.Close()
        return out

    # every e2e step is timed on its own (wall clock around the public API call, which ends with the
    # device->host read of the result); the MEDIAN step is reported: the host part (Python, id maps,
    # pinned copies) is exposed to noisy neighbours on these shared boxes, the device part is not
    e2e_steps = args.steps
    step_e2e()
    barrier()
    e2e_times = []
    for _ in range(e2e_steps):
        barrier()
        t0 = time.perf_counter()
        step_e2e()
        torch.cuda.synchronize()
        e2e_times.append(time.perf_counter() - t0)
    e2e_s = statistics.median(e2e_times)

    # ---- reduce over ranks: max time, summed units ----
    pairs_full = n_left * (n_left - 1) / 2.0
    if world > 1 and args.folds:
        pairs_rank = pairs_full                                  # a fold per GPU
    elif shard:
        pairs_rank = (re - rb) * (n_left - 1) / 2.0
    else:
        pairs_rank = pairs_full / (world if multi else 1)        # every pair once across the ranks
    red = torch.tensor([total_ms, e2e_s, prof["sim_kernel_ms"], prof["predict_kernel_ms"], prof["prep_ms"]],
                       dtype=torch.float64, device=dev)
    units = torch.tensor([pairs_rank, float(n_mine_cyc if cyc else n_pred)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
        dist.all_reduce(units, op=dist.ReduceOp.SUM)
    total_ms, e2e_s, sim_ms, pred_ms, prep_ms = red.tolist()
    pairs_all, preds_all = units.tolist()
    if rank != 0:
        h.close()
        return

    ms_per_step = total_ms / args.steps
    value = pairs_all / (ms_per_step / 1e3)
    hbm_peak, peak_src = load_peaks()
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
    # dominant kernel = the similarity kernel.  Algorithmic bytes per launch (DESIGN.md §Kernels):
    # one read of the left CSR (4 B id + 8 B rating per entry) + 8 B per similarity the kernel emits
    # (the computed triangle; the mirror pass writes the rest) — stream path; the tensor path
    # reports int8 ops instead.
    sim_launch_ms = sim_ms / max(1, prof["sim_launches"])
    launches_per_step = max(1, prof["sim_launches"]) / args.steps
    sim_step_ms = sim_ms / args.steps            # all similarity launches of one Fit (slabs in top-k mode)
    # cuBLASLt's sustained figure is what the box delivers after seconds of tensor load (power-capped clocks);
    # a Fit whose tensor kernels run for less than half a second never gets there and is held to the burst figure
    tpeak, tpeak_src = int8_peak(peaks, peak_src, long_kernel=sim_step_ms > 500.0)
    g = {"cosine": 3, "msd": 4, "pearson": 6, "pearson_baseline": 6, "slope_one": 3}[sim]   # slope one: count, sum r_i, sum r_j
    dense_ops = pairs_rank * 2 * g * n_right
    if prof["sim_path_used"] == rs.core.RS_SIM_PATH["tensor"]:
        roof = {"bound": "tensor", "achieved": dense_ops / (sim_step_ms / 1e3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                "frac": dense_ops / (sim_step_ms / 1e3) / 1e12 / tpeak, "traffic": None,
                "peak_source": tpeak_src,
                "kernel": ("sim_tensor_pair_kernel" if sim in ("cosine", "msd") and
                           (n_left / 128.0) * (n_left / 128.0) / 2 >= 4 * 148 else "sim_tensor_kernel"),
                "ms_per_launch": sim_launch_ms,
                "launches_per_step": launches_per_step,
                "note": ("algorithmic int8 ops of the rank's unordered pairs / time of all similarity launches of "
                         "one Fit" + ("; a row shard computes full rows (2x the algorithmic ops) and the time "
                                      "includes the per-slab top-k selection" if shard else
                                      "; includes the per-slab transpose and top-k merges" if sym else ""))}
    else:
        emitted = pairs_rank + (n_left / (world if multi else 1))   # the computed triangle + the diagonal
        alg_bytes = len(left) * 12 + emitted * 8
        roof = {"bound": "hbm", "achieved": alg_bytes / (sim_step_ms / 1e3) / 1e9, "peak": hbm_peak,
                "unit": "GB/s", "frac": alg_bytes / (sim_step_ms / 1e3) / 1e9 / hbm_peak, "traffic": None,
                "peak_source": f"{peak_src} copy bandwidth", "kernel": f"sim_stream_kernel<{sim}>",
                "ms_per_launch": sim_launch_ms, "launches_per_step": launches_per_step,
                "triples_per_sec": prof["corated_triples"] / (world if multi else 1) / (sim_step_ms / 1e3),
                "dense_equivalent": {"tops": dense_ops / (sim_step_ms / 1e3) / 1e12, "int8_peak_tops": tpeak,
                                     "frac": dense_ops / (sim_step_ms / 1e3) / 1e12 / tpeak,
                                     "note": ("int8 ops the dense masked-contraction formulation of the same pairs "
                                              "needs (SURVEY.md §8d: N(N-1)/2 * 2*G*K) / this kernel's time, against "
                                              "the int8 tensor roofline: > 1 means the exact sparse replay finishes "
                                              "before a tensor-core kernel running AT its roofline could")},
                "note": ("exact-order FP64 sparse replay: work = the co-rated triples; bound by shared-memory "
                         "read-modify-write wavefronts and issue slots, not by HBM (profiles/r02_stream_notes.md); "
                         "reported against the HBM roofline of its algorithmic bytes (left CSR + emitted "
                         "similarities) as the contract asks")}
    # second object for the gather-reduce (the north star asks for "achieved HBM GB/s for predict"):
    # algorithmic bytes per prediction (SURVEY.md §8d) = C * (4 B id + 1 B rating + 8 B similarity
    # [+ 8 B mean/bias for the non-basic types]) + 8 B out
    roof_pred = None
    if n_pred:
        deg_right = np.bincount(right, minlength=n_right)
        t_right_own = t_right[own_cyc] if cyc else t_right          # the pairs THIS rank's kernel answered
        cand = float(deg_right[t_right_own[t_right_own >= 0]].sum())
        per_cand = 13 + (8 if knn_type != "basic" else 0)
        n_answered = n_mine_cyc if cyc else n_pred
        pbytes = cand * per_cand + n_answered * 8.0
        pms = pred_ms / args.steps
        roof_pred = {"bound": "hbm", "achieved": pbytes / (pms / 1e3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": pbytes / (pms / 1e3) / 1e9 / hbm_peak, "traffic": None,
                     "kernel": "predict_select_kernel", "ms_per_launch": pms,
                     "bytes_per_candidate": per_cand,
                     "candidates_per_prediction": cand / max(1, n_answered)}
    prof_file = ROOT / "profiles" / "traffic.json"
    if prof_file.exists():
        try:
            # DRAM bytes per launch of this kernel ON THIS WORKLOAD from the committed ncu capture
            tj = json.loads(prof_file.read_text())
            if world == 1:
                roof["traffic"] = tj.get(roof["kernel"].split("<")[0] + "|" + args.workload)
                if roof_pred:
                    roof_pred["traffic"] = tj.get("predict_select_kernel|" + args.workload)
        except (ValueError, OSError):
            pass

    parallelism = ("single GPU" if world == 1 else
                   "one fold per GPU, no collective" if args.folds else
                   "symmetric slabs dealt in snake order + NCCL all-gather and union of partial neighbour lists" if sym else
                   "cyclic row shards: every pair once, other triangle pulled from peer memory over NVLink "
                   "(CUDA IPC), every shard answers the test pairs of its rows, NCCL all-reduce (int64 sum of the bit "
                   "patterns) assembles the predictions" if cyc else
                   "contiguous row shards (full rows) + NCCL all-gather of neighbour lists")
    limiter = None
    if multi:
        fixed = prep_ms / args.steps
        rest = ms_per_step - (sim_ms + pred_ms + prep_ms) / args.steps
        limiter = (f"(1) replicated per-rank work: the CSR build, {fixed:.1f} ms of the {ms_per_step:.1f} ms step, is not "
                   f"divided by N (every rank sorts the full rating set); (2) the exchange step (mirror over NVLink, two "
                   f"small collectives, the all-reduce of the predictions) and launch gaps: {rest:.1f} ms; the similarity "
                   f"kernel ({sim_ms / args.steps:.1f} ms) and Predict ({pred_ms / args.steps:.1f} ms) are divided by N")
    line = {
        "metric": "similarity_pairs_per_sec", "value": value, "unit": "pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if multi else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "predictions_per_sec": preds_all / (ms_per_step / 1e3),
        "config": {"workload": args.workload, "shape": f"{users}x{items}", "train_ratings": train.Length(),
                   "test_pairs": int(preds_all), "sim": sim, "knn_type": knn_type, "user_based": user_based, "k": k,
                   "tie_policy": "canonical", "pearson_mode": args.pearson_mode,
                   "sim_path": {0: "auto", 1: "tensor", 2: "stream"}[prof["sim_path_used"]],
                   "l2": "flushed between timed iterations (256 MiB write)",
                   "parallelism": parallelism},
        "clocks": clock_info,
        "e2e": {"value": pairs_all / e2e_s, "unit": "pairs/s", "ms_per_step": e2e_s * 1e3,
                "h2d_bytes_per_step": int(len(left) * 16 / (world if cyc else 1) + test.Length() * 8),
                "d2h_bytes_per_step": int(n_pred * 8 + (n_left * k * 12 if sym else 0)),
                "predictions_per_sec": preds_all / e2e_s, "steps": e2e_steps, "statistic": "median step",
                "ms_min": min(e2e_times) * 1e3, "ms_max": max(e2e_times) * 1e3},
        "gpu_launches": int(prof["total_launches"]),
        "kernel_ms": {"sim": sim_ms / args.steps, "predict": pred_ms / args.steps, "prep": prep_ms / args.steps},
        "corated_triples": prof["corated_triples"],
        "roofline": roof,
        "roofline_predict": roof_pred,
    }
    if limiter:
        line["scaling_limiter"] = limiter
    if world == 1 and not args.no_cpu_baseline:
        from oracle import binding as ob

        ots = ob.TrainSet(train.Users, train.Items, train.Ratings)
        cores = os.cpu_count() or 1
        n = n_left
        # >= 24 rows per host thread: the reference's static row split (core/knn.go:192-199) is badly balanced on fewer
        slab = representative_slab(left, n, cpu_sample_rows(n, train.Length(), 1.8e10))
        tf, tp, rows_done, npred = cpu_reference_step(ob, ots, test, sim, knn_type, user_based, k, cores,
                                                      rows=slab, n_pred=20000)
        # slab: rows_done x (n-1) ordered pairs; the full Fit computes each unordered pair about once
        est_fit = tf * (n / rows_done) * 0.5
        if rows_done >= n:
            est_fit = tf
            sample = f"full Fit ({n} rows, {cores} threads) + first {npred} test pairs predicted serially"
        elif est_fit < 25:
            tf, tp, rows_done, npred = cpu_reference_step(ob, ots, test, sim, knn_type, user_based, k, cores,
                                                          n_pred=20000)
            est_fit = tf
            sample = f"full Fit ({n} rows, {cores} threads) + first {npred} test pairs predicted serially"
        else:
            sample = (f"Fit slab of rows [{slab[0]},{slab[1]}) (mean row length closest to the matrix mean) x all {n} "
                      f"({cores} threads, scaled x{n / rows_done:.1f}/2) + first {npred} of the slab's test pairs "
                      f"predicted serially")
        cpu_step = est_fit + (tp / max(1, npred)) * test.Length()
        line["cpu_baseline"] = {"value": (n * (n - 1) / 2) / cpu_step, "unit": "pairs/s", "cores": cores,
                                "kind": "port", "sample": sample, "fit_s": est_fit,
                                "predict_s": (tp / max(1, npred)) * test.Length()}
    print(json.dumps(line), flush=True)
    h.close()


def int8_peak(peaks, peak_src, long_kernel=False):
    """Denominator of the tensor roofline: the measured plain dense int8 GEMM peak when profiles/ holds one
    (tools/i8_peak.py, SURVEY.md §7.3 item 5) — the burst figure for a kernel timed alone, the sustained one
    for a Fit that keeps the tensor cores busy for more than half a second —, else 2 x the measured bf16 burst,
    labelled."""
    f = ROOT / "profiles" / "int8_peak.json"
    if f.exists():
        try:
            j = json.loads(f.read_text())
            key = "tops_sustained" if long_kernel else "tops"
            return float(j[key]), f"measured dense int8 GEMM, {key} ({j.get('how', 'tools/i8_peak.py')})"
        except (ValueError, KeyError, OSError):
            pass
    return 2.0 * float(peaks.get("bf16_tflops", 1590.0)), f"2 x {peak_src} bf16 burst (no measured int8 peak committed)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--shard-rows", action="store_true", help="N > 1: contiguous row shards even on the exact sparse path")
    ap.add_argument("--folds", action="store_true", help="N > 1: one cross-validation fold per GPU (weak scaling), "
                    "the reference's own parallelism (core/eval.go:28-35)")
    ap.add_argument("--pearson-mode", default="exact", choices=["exact", "sums"])
    ap.add_argument("--sim-path", default="auto", choices=["auto", "tensor", "stream"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64, under 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl")
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
