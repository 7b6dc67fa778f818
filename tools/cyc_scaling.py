#!/usr/bin/env python
"""Per-shard time of the exact sparse Fit under cyclic row sharding, measured on ONE GPU: fits shard 0
of `count` shards (no peers needed for the similarity kernel itself) and prints the kernel time.
usage: [CYC_INDEX=i] tools/cyc_scaling.py [workload] [counts...]"""
import os
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402
import recommend_sys_b200 as rs  # noqa: E402
import torch  # noqa: E402

wl = sys.argv[1] if len(sys.argv) > 1 else "ml20m_item_pearson_k40"
counts = [int(x) for x in sys.argv[2:]] or [1, 2, 4, 8]
users, items, nnz, n_test, sim, knn_type, user_based, k = bench.WORKLOADS[wl]
train, test = bench.make_data(wl)
n_left = train.UserCount if user_based else train.ItemCount
n_right = train.ItemCount if user_based else train.UserCount
left = train.innerUsers if user_based else train.innerItems
right = train.innerItems if user_based else train.innerUsers
dev = torch.device("cuda", 0)
d_left, d_right = torch.from_numpy(left).to(dev), torch.from_numpy(right).to(dev)
d_rating = torch.from_numpy(train.Ratings).to(dev)
# CYC_SWEEP="min:max,min:max,...": popular-column thresholds (RS_KNN_POP_MIN : RS_KNN_POP_MAX) to run in one process
sweep = [x.split(":") for x in os.environ["CYC_SWEEP"].split(",")] if "CYC_SWEEP" in os.environ else [None]
for sw, count in [(s_, c_) for s_ in sweep for c_ in counts]:
    if sw:
        os.environ["RS_KNN_POP_MIN"], os.environ["RS_KNN_POP_MAX"] = sw
        print("threshold", sw, end=" ")
    for index in ([int(os.environ["CYC_INDEX"])] if "CYC_INDEX" in os.environ else sorted({0, count - 1})):
        h = rs.core._Handle(sim=sim, knn_type=knn_type, k=k, device=0, shard_count=count if count > 1 else 0,
                            shard_index=index, sim_path="stream")
        ms = []
        for rep in range(4):
            h.profile_reset()
            h.fit_device(d_left.data_ptr(), d_right.data_ptr(), d_rating.data_ptr(), len(left), n_left, n_right,
                         train.GlobalMean)
            p = h.profile()
            ms.append(p["sim_kernel_ms"])
        print(f"{wl} shards={count} index={index} sim_ms={min(ms[1:]):.2f} prep_ms={p['prep_ms']:.2f}", flush=True)
        h.close()
