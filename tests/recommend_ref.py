"""Restatement of top-N recommendation on the host (include/rs_knn.h, rs_knn_score_all / rs_knn_recommend).

score_all loops every target of a query through the oracle's canonical-tie Predict and sets the targets the query
rated to NaN; rank_rows applies the ranking rule: NaN never listed, (score desc, target id asc), +-0 tie by id and
keep their sign, unused slots id -1 / score NaN."""
import numpy as np


def raw_by_inner(raw):
    """Raw ids in inner-id order (inner id = order of first appearance, core/data.go:137-151)."""
    _, first = np.unique(raw, return_index=True)
    return raw[np.sort(first)]


def inner_of(raw):
    table = {v: n for n, v in enumerate(raw_by_inner(raw).tolist())}
    return np.array([table[v] for v in raw.tolist()], dtype=np.int64)


def score_all(ref, u, i, user_based, side, queries):
    """Oracle score rows [len(queries)][n_targets] over inner ids; side "left" / "right" as in rs_knn.h."""
    users, items = raw_by_inner(u), raw_by_inner(i)
    left_raw, right_raw = (users, items) if user_based else (items, users)
    lu, ri = (inner_of(u), inner_of(i)) if user_based else (inner_of(i), inner_of(u))
    q_raw, t_raw = (left_raw, right_raw) if side == "left" else (right_raw, left_raw)
    queries = np.asarray(queries, dtype=np.int64)
    nt = len(t_raw)
    qq = np.repeat(queries, nt)
    tt = np.tile(np.arange(nt), len(queries))
    l_ids, r_ids = (qq, tt) if side == "left" else (tt, qq)
    lr = np.where(l_ids >= 0, left_raw[np.maximum(l_ids, 0)], -(1 << 40))     # -1 -> an id the oracle never saw
    rr = np.where(r_ids >= 0, right_raw[np.maximum(r_ids, 0)], -(1 << 40))
    pu, pi = (lr, rr) if user_based else (rr, lr)
    out = ref.predict_batch(pu, pi, n_threads=8).reshape(len(queries), nt)
    rated = {}
    for l, r in zip(lu.tolist(), ri.tolist()):
        q, t = (l, r) if side == "left" else (r, l)
        rated.setdefault(q, []).append(t)
    for b, q in enumerate(queries.tolist()):
        if q >= 0:
            out[b, rated[q]] = np.nan
    return out


def rank_rows(scores, n_top):
    """(ids, scores) [rows][n_top] of the ranking rule."""
    rows = scores.shape[0]
    ids = np.full((rows, n_top), -1, dtype=np.int32)
    top = np.full((rows, n_top), np.nan)
    for b in range(rows):
        s = scores[b]
        valid = np.flatnonzero(~np.isnan(s))
        order = valid[np.lexsort((valid, -(s[valid] + 0.0)))][:n_top]
        ids[b, :len(order)] = order
        top[b, :len(order)] = s[order]
    return ids, top


def same_bits(a, b):
    """Bit-identical, any NaN equal to any NaN."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64),
                                                                            b[~nb].view(np.uint64))
