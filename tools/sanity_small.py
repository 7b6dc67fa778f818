"""Small end-to-end exercise of every kernel family (for compute-sanitizer runs on the GPU box):
    compute-sanitizer --tool memcheck python tools/sanity_small.py
Checks results against the oracle as it goes."""
import os
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np

import recommend_sys_b200 as rs
from oracle import binding as ob

data = rs.core.synth_ratings(500, 700, 30000, 0x5EED0000)
n_test = 3000
train = rs.NewTrainSet(data.SubSet(np.arange(n_test, data.Length())))
test = data.SubSet(np.arange(0, n_test))


def fresh_ots():
    # a new oracle TrainSet per fit: like the reference, the oracle's KNN.Fit sorts the cached adjacency
    # lists in place (core/data.go:236-243), which changes the 'dataset order' a later z-score fit sees
    return ob.TrainSet(train.Users, train.Items, train.Ratings)


def same(a, b):
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.nan_to_num(a, posinf=1e300, neginf=-1e300),
                                                                      np.nan_to_num(b, posinf=1e300, neginf=-1e300))


cases = [("msd", "basic", True, {"simPath": "tensor"}, {"RS_KNN_TC_PAIR": "1"}),
         ("cosine", "basic", False, {"simPath": "tensor"}, {"RS_KNN_TC_PAIR": "0"}),
         ("pearson", "centered", False, {}, {}),
         ("msd", "zscore", True, {"simPath": "stream"}, {"RS_KNN_STREAM_JC": "256"}),
         ("pearson_baseline", "baseline", False, {"baseline": "als", "shrinkage": 50.0}, {})]
SIM = {"msd": rs.MSD, "cosine": rs.Cosine, "pearson": rs.Pearson, "pearson_baseline": rs.PearsonBaseline}
CT = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore, "baseline": rs.NewKNNBaseLine}
for sim, typ, ub, extra, env in cases:
    for k_, v_ in env.items():
        os.environ[k_] = v_
    p = {"sim": SIM[sim], "userBased": ub, "k": 40}
    p.update(extra)
    est = CT[typ](rs.Parameters(p))
    est.Fit(train)
    got = test.Predict(est)
    ref = ob.KNN(sim=sim, knn_type=typ, user_based=ub, k=40, baseline=extra.get("baseline", "sgd"),
                 shrinkage=extra.get("shrinkage", 0.0)).fit(fresh_ots())
    assert same(est.Sims, ref.sims()), (sim, typ, "sims")
    assert same(got, ref.predict_batch(test.Users, test.Items)), (sim, typ, "predictions")
    print("ok", sim, typ, ub, extra, env, flush=True)
    est.Close()
    for k_ in env:
        os.environ.pop(k_, None)

# Pearson sums mode (tensor) + integer co-rating sums
est = rs.NewKNN(rs.Parameters({"sim": rs.Pearson, "userBased": False, "pearsonMode": "sums", "simPath": "tensor"}))
est.Fit(train)
ref = ob.KNN(sim="pearson", user_based=False).fit(fresh_ots())
S, W = est.Sims, ref.sims()
ok = ~np.isnan(W)
assert np.array_equal(np.isnan(S), np.isnan(W)) and (np.abs(S[ok] - W[ok]) <= 1e-9 * np.maximum(1, np.abs(W[ok]))).all()
est._h.cosums(0, 4)
print("ok pearson sums + cosums", flush=True)
est.Close()

# symmetric slabs, 3 shards, union
import torch

from recommend_sys_b200.shard import union_topk_device

os.environ["RS_KNN_SLAB_ROWS"] = "256"
full = rs.NewKNN(rs.Parameters({"sim": rs.MSD, "userBased": True}))
full.Fit(train)
wi, ws = full.TopK(30)
parts = []
for r in range(3):
    pz = rs.NewKNN(rs.Parameters({"sim": rs.MSD, "userBased": True, "store": "topk", "topk": 30, "shardCount": 3,
                                  "shardIndex": r}))
    pz.Fit(train)
    parts.append(pz.TopK(30))
    pz.Close()
ai = torch.from_numpy(np.stack([a for a, _ in parts])).cuda()
as_ = torch.from_numpy(np.stack([b for _, b in parts])).cuda()
ui, us = union_topk_device(ai, as_)
torch.cuda.synchronize()
assert np.array_equal(ui.cpu().numpy(), wi) and same(us.cpu().numpy(), ws)
print("ok symmetric slabs", flush=True)
