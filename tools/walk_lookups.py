#!/usr/bin/env python
"""(entry, chunk) lookups of the exact sparse column walk when popular columns are split off, counted on the CPU
for a bench workload.  Row i of the walk pays one lookup per entry and per JC-column chunk it visits; a lookup is
non-empty when c's run in that chunk holds a partner.  Counted with the walked rows' columns at their first-appearance
ids (the layout before labels) and at their labels (rank in the stable longest-first order of all rows minus the
popular rows, prep.cu split_popular), for the lower triangle; the upper triangle's lookups decide between them.
usage: tools/walk_lookups.py [workload] [--jc 256] [--pop-min 8192] [--pop-max 512]"""
import argparse
import sys
from pathlib import Path

import numpy as np


def ranks(deg):
    """position of every row in the stable longest-first order (ties by ascending id)"""
    order = np.argsort(-deg, kind="stable")
    rank = np.empty(len(deg), np.int64)
    rank[order] = np.arange(len(deg))
    return rank


def popular_count(deg, pop_min, pop_max):
    """rows split off as popular columns: those of >= pop_min entries, at most pop_max; fewer than 2: none"""
    n = min(int((deg >= pop_min).sum()), pop_max)
    return n if n >= 2 else 0


def count(left, right, col, walk, n_cols, jc):
    """lookups of the lower (j < i) and upper triangle, non-empty lookups and co-rated triples of the lower one.
    left / right: the rows and right ids of the ratings; col[i]: row i's column in the walk, of n_cols; walk[i]: i is
    walked."""
    deg = np.bincount(left, minlength=len(col))
    n_q = (n_cols + jc - 1) // jc
    q = col // jc
    lower = int((deg[walk] * (q[walk] + 1)).sum())
    upper = int((deg[walk] * (n_q - q[walk])).sum())
    keep = walk[left]
    ck, rk = col[left[keep]], right[keep]
    o = np.lexsort((ck, rk))
    ck, rk = ck[o], rk[o]
    if len(rk) == 0:
        return lower, upper, 0, 0
    start = np.r_[True, rk[1:] != rk[:-1]]
    ch = ck // jc
    newch = start | np.r_[True, ch[1:] != ch[:-1]]
    grp = np.cumsum(start) - 1
    first = np.flatnonzero(start)[grp]
    cs = np.cumsum(newch)
    nonempty = int((cs - cs[first] + 1 - newch).sum())     # chunks holding an earlier entry of the same right id
    triples = int((np.arange(len(rk)) - first).sum())      # earlier entries of the same right id
    return lower, upper, nonempty, triples


def layouts(left, n_left, pop_min, pop_max):
    """n_pop and (name, col, walk, n_cols) of the two layouts: first-appearance ids (chunks over all rows) and labels
    (chunks over the walked rows)"""
    deg = np.bincount(left, minlength=n_left)
    rank = ranks(deg)
    n_pop = popular_count(deg, pop_min, pop_max)
    walk = rank >= n_pop
    return n_pop, [("first-appearance id", np.arange(n_left), walk, n_left),
                   ("label (longest first)", rank - n_pop, walk, n_left - n_pop)]


def main():
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    import bench

    ap = argparse.ArgumentParser()
    ap.add_argument("workload", nargs="?", default=bench.DEFAULT_WORKLOAD, choices=sorted(bench.WORKLOADS))
    ap.add_argument("--jc", type=int, default=256)
    ap.add_argument("--pop-min", type=int, default=8192)
    ap.add_argument("--pop-max", type=int, default=512)
    args = ap.parse_args()
    user_based = bench.WORKLOADS[args.workload][6]
    train, _ = bench.make_data(args.workload)
    left = np.asarray(train.innerUsers if user_based else train.innerItems, np.int64)
    right = np.asarray(train.innerItems if user_based else train.innerUsers, np.int64)
    n_left = int(left.max()) + 1
    n_pop, lays = layouts(left, n_left, args.pop_min, args.pop_max)
    print(f"{args.workload}: rows {n_left}, popular {n_pop}, walked {n_left - n_pop}, jc {args.jc}")
    print(f"{'walked rows ordered by':24s} {'lookups':>11s} {'non-empty':>11s} {'triples':>11s} "
          f"{'triples/lookup':>14s} {'upper lookups':>14s}")
    for name, col, walk, n_cols in lays:
        lo, up, ne, tr = count(left, right, col, walk, n_cols, args.jc)
        print(f"{name:24s} {lo:11.4e} {ne:11.4e} {tr:11.4e} {tr / max(lo, 1):14.2f} {up:14.4e}")


if __name__ == "__main__":
    main()
