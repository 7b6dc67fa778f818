"""Host restatement of top-N recommendation (tests/recommend_ref.py), checked without a GPU."""
import math
import struct

import numpy as np

from oracle import binding as ob
from recommend_ref import rank_rows, raw_by_inner, same_bits, score_all


def _sim_key(s):
    """rs_sim_key (csrc/common.cuh): order-preserving 64-bit key, -0.0 folded to +0.0."""
    b = struct.unpack("<Q", struct.pack("<d", s + 0.0))[0]
    return (~b & (2 ** 64 - 1)) if b >> 63 else b | (1 << 63)


def test_rank_rows_follows_the_ranking_rule():
    rng = np.random.RandomState(3)
    pool = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.5, -1.5, 2.0, 1e-300, -1e-300])
    for n_top in (1, 3, 10, 40):
        s = pool[rng.randint(0, len(pool), (20, 30))]
        ids, top = rank_rows(s, n_top)
        for b in range(s.shape[0]):
            order = sorted((t for t in range(s.shape[1]) if not math.isnan(s[b, t])),
                           key=lambda t: (-_sim_key(s[b, t]), t))[:n_top]
            assert ids[b, :len(order)].tolist() == order
            assert (ids[b, len(order):] == -1).all() and np.isnan(top[b, len(order):]).all()
            assert same_bits(top[b, :len(order)], s[b, order])          # -0.0 stays -0.0


def test_score_all_is_predict_with_rated_targets_nan():
    rng = np.random.RandomState(5)
    u = rng.randint(0, 30, 400).astype(np.int64)
    i = rng.randint(0, 25, 400).astype(np.int64)
    keep = np.unique(u * 1000 + i, return_index=True)[1]
    u, i = u[keep], i[keep]
    r = rng.randint(1, 6, len(u)).astype(np.float64)
    for user_based in (True, False):
        ref = ob.KNN(sim="pearson", knn_type="centered", user_based=user_based, k=5, min_k=1,
                     tie_policy="canonical").fit(ob.TrainSet(u, i, r))
        users, items = raw_by_inner(u), raw_by_inner(i)
        side = "left" if user_based else "right"
        q = np.array([0, 3, -1, 7])
        got = score_all(ref, u, i, user_based, side, q)
        rated = set(zip(u.tolist(), i.tolist()))
        for b, qq in enumerate(q.tolist()):
            for t, item in enumerate(items.tolist()):
                if qq < 0:
                    assert got[b, t] == ref.global_mean()
                    continue
                user = users[qq]
                if (user, item) in rated:
                    assert math.isnan(got[b, t])
                else:
                    assert same_bits([got[b, t]], [ref.predict(user, item)])
