#!/usr/bin/env python
"""Diagnostic for the popular-column split of the exact sparse Fit (sim_stream.cu: the dense items of
sim_stream_kernel): fits ml-100k with a low threshold and reports, per class of cell (popular x popular, other x
popular, popular x other, other x other), how many cells differ from the oracle.
usage: tools/pop_diag.py [pop_min] [sim] [user_based 0|1]"""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import recommend_sys_b200 as rs  # noqa: E402
from oracle import binding as ob  # noqa: E402

pop_min = sys.argv[1] if len(sys.argv) > 1 else "150"
sim = sys.argv[2] if len(sys.argv) > 2 else "pearson"
user_based = bool(int(sys.argv[3])) if len(sys.argv) > 3 else False
os.environ["RS_KNN_POP_MIN"] = pop_min
g = np.load(ROOT / "tests" / "golden" / "ml100k.npz")
a = g["u2_base"].astype(np.int64)
u, i, r = a[:, 0], a[:, 1], a[:, 2].astype(np.float64)
SIMS = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson}
ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
for tri in ("lower", "upper"):
    os.environ["RS_KNN_STREAM_TRI"] = tri
    est = rs.NewKNN(rs.Parameters({"sim": SIMS[sim], "userBased": user_based, "k": 40, "simPath": "stream"}))
    est.Fit(ts)
    got = est.Sims
    ref = ob.KNN(sim=sim, knn_type="basic", user_based=user_based, k=40, n_jobs=8, tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    want = ref.sims()
    left = ts.innerUsers if user_based else ts.innerItems
    n = want.shape[0]
    cnt = np.bincount(left, minlength=n)
    order = np.argsort(-cnt, kind="stable")
    n_pop = min(int((cnt >= int(pop_min)).sum()), 512)
    pop = np.zeros(n, bool)
    pop[order[:n_pop]] = True
    ng, nw = np.isnan(got), np.isnan(want)
    bad = (ng != nw) | (~ng & ~nw & (got.view(np.uint64) != want.view(np.uint64)))
    print(f"tri={tri} pop_min={pop_min} sim={sim} user_based={user_based} n={n} n_pop={n_pop} bad cells={int(bad.sum())}")
    for name, rm, cm in (("pop x pop", pop, pop), ("other x pop", ~pop, pop), ("pop x other", pop, ~pop), ("other x other", ~pop, ~pop)):
        sub = bad[np.ix_(rm, cm)]
        lo = np.tril(np.ones((n, n), bool), -1)[np.ix_(rm, cm)]
        print(f"  {name:14s} cells={sub.size:9d} bad={int(sub.sum()):9d} (below diag {int((sub & lo).sum())}, above {int((sub & ~lo).sum())})"
              f" got-NaN-where-want-finite={int((ng & ~nw)[np.ix_(rm, cm)].sum())} want-NaN-got-finite={int((~ng & nw)[np.ix_(rm, cm)].sum())}")
    if bad.any():
        rr, cc = np.nonzero(bad)
        for k in range(min(8, len(rr))):
            print(f"    ({rr[k]},{cc[k]}) pop=({pop[rr[k]]},{pop[cc[k]]}) got={got[rr[k], cc[k]]!r} want={want[rr[k], cc[k]]!r}")
    est.Close()
