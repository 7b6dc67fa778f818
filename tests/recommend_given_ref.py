"""Host restatement of top-N recommendation for queries given as rating lists (include/rs_knn.h,
rs_knn_score_all_given / rs_knn_recommend_given).

A list is (inner ids of the target side, ratings) in the caller's order.
  right side (item-based): the candidates of every target t are the list's entries in ascending id, weighted by the
    fitted row S[t] (or_knn_sims_row); their statistics are the fitted ones.
  left side (user-based): S*[v] = or_sim_lists(list sorted by or_sort_by_id, L(v)) for every fitted left row v; the
    candidates of target t are its fitted raters R(t), weighted by S*; the query's mean / stddev are summed in the
    caller's order (core/knn.go:167-177).
The canonical Predict (core/knn.go:93-141, ties by ascending id) is restated with sequential float64 sums, vectorised
over the targets; the list's ids are then NaN, and recommend_ref.rank_rows ranks the rows."""
import math

import numpy as np

from oracle import binding as ob
from recommend_ref import inner_of, raw_by_inner

KNN_TYPES = ("basic", "centered", "zscore", "baseline")


class Model:
    """The fitted state the restatement reads, over inner ids: an oracle KNN fitted on (u, i, r)."""

    def __init__(self, u, i, r, sim, knn_type, user_based, k=40, min_k=1):
        self.sim, self.knn_type, self.user_based, self.k, self.min_k = sim, knn_type, user_based, k, min_k
        self.ref = ob.KNN(sim=sim, knn_type=knn_type, user_based=user_based, k=k, min_k=min_k, n_jobs=8,
                          tie_policy="canonical").fit(ob.TrainSet(u, i, r))
        iu, ii = inner_of(np.asarray(u)), inner_of(np.asarray(i))
        left, right = (iu, ii) if user_based else (ii, iu)
        r = np.asarray(r, dtype=np.float64)
        self.n_left, self.n_right = int(left.max()) + 1, int(right.max()) + 1
        self.sims = self.ref.sims()
        self.means, self.stddevs, self.bias = self.ref.means(), self.ref.stddevs(), self.ref.bias()
        self.global_mean = self.ref.global_mean()
        # R(t): the raters of each right row, ascending left id, padded with -1
        order = np.lexsort((left, right))
        counts = np.bincount(right, minlength=self.n_right)
        width = max(1, int(counts.max()))
        self.r_ids = np.full((self.n_right, width), -1, dtype=np.int64)
        self.r_val = np.full((self.n_right, width), np.nan)
        start = np.concatenate([[0], np.cumsum(counts)[:-1]])
        pos = np.arange(len(order)) - np.repeat(start, counts)
        self.r_ids[right[order], pos] = left[order]
        self.r_val[right[order], pos] = r[order]
        # L(v): each left row as the oracle's sorted (id, rating) list, for or_sim_lists
        self._rows = []
        by_left = np.argsort(left, kind="stable")
        bounds = np.concatenate([[0], np.cumsum(np.bincount(left, minlength=self.n_left))])
        for v in range(self.n_left):
            sel = by_left[bounds[v]:bounds[v + 1]]
            self._rows.append(_id_ratings(right[sel], r[sel]))

    def given_sims(self, ids, vals):
        """S*[v] = Sim(list sorted by id, L(v)) for every fitted left row v."""
        a, na = _id_ratings(ids, vals)
        L = ob.lib()
        code = ob.SIM[self.sim]
        return np.array([L.or_sim_lists(code, a, na, b, n) for b, n in self._rows])

    def score_given(self, side, ids, vals):
        """One score row of the list (ids, vals) in the caller's order."""
        ids = np.asarray(ids, dtype=np.int64)
        vals = np.asarray(vals, dtype=np.float64)
        if side == "right":
            o = np.argsort(ids, kind="stable")
            cid, cval = ids[o], vals[o]
            nt = self.n_left
            s = self.sims[:, cid]
            c_ids = np.broadcast_to(cid, s.shape)
            c_val = np.broadcast_to(cval, s.shape)
            t = np.arange(nt)
            lmean = self.means[t] if self.means is not None else None
            lstd = self.stddevs[t] if self.stddevs is not None else None
            lbias = self.bias[t] if self.bias is not None else None
        else:
            nt = self.n_right
            star = self.given_sims(ids, vals)
            c_ids, c_val = self.r_ids, self.r_val
            s = np.where(c_ids >= 0, star[np.maximum(c_ids, 0)], np.nan)
            lmean, lstd = list_stats(vals)
            lbias = None
        out = self._predict(s, c_ids, c_val, lmean, lstd, lbias, nt)
        out[ids] = np.nan
        return out

    def _predict(self, s, c_ids, c_val, lmean, lstd, lbias, nt):
        gm = self.global_mean
        if s.shape[1] == 0:
            return np.full(nt, gm)
        valid = ~np.isnan(s)
        nvalid = valid.sum(axis=1)
        key = np.where(valid, -s, np.inf)                  # similarity desc, NaN last; +-0 tie, then id asc
        order = np.lexsort((c_ids, key), axis=-1)
        ss = np.take_along_axis(s, order, axis=-1)
        sid = np.maximum(np.take_along_axis(np.asarray(c_ids), order, axis=-1), 0)
        rating = np.take_along_axis(np.asarray(c_val), order, axis=-1)
        with np.errstate(all="ignore"):
            if self.knn_type == "centered":
                rating = rating - self.means[sid]
            elif self.knn_type == "zscore":
                rating = (rating - self.means[sid]) / self.stddevs[sid]
            elif self.knn_type == "baseline":
                rating = rating - self.bias[sid]
            num = np.minimum(nvalid, self.k)
            wsum = np.zeros(nt)
            wrat = np.zeros(nt)
            for x in range(min(self.k, s.shape[1])):         # core/knn.go:116-130, one neighbour at a time
                on = x < num
                wsum = np.where(on, wsum + ss[:, x], wsum)
                wrat = np.where(on, wrat + ss[:, x] * rating[:, x], wrat)
            pred = wrat / wsum                                # core/knn.go:131-140
            if self.knn_type == "centered":
                pred = pred + lmean
            elif self.knn_type == "baseline":
                pred = pred + lbias
            elif self.knn_type == "zscore":
                pred = pred * lstd
                pred = pred + lmean
        return np.where(nvalid <= self.min_k, gm, pred)

    def score_all_given(self, side, ptr, ids, vals):
        return np.stack([self.score_given(side, ids[ptr[b]:ptr[b + 1]], vals[ptr[b]:ptr[b + 1]])
                         for b in range(len(ptr) - 1)])


def _id_ratings(ids, vals):
    """An oracle (id, rating) list sorted by or_sort_by_id (the reference's sorts, core/data.go:249)."""
    n = len(ids)
    a = (ob.IdRating * max(1, n))(*[ob.IdRating(int(x), float(y)) for x, y in zip(ids, vals)])
    ob.lib().or_sort_by_id(a, n)
    return a, n


def list_stats(vals):
    """The list's mean and stddev, summed in the caller's order (core/data.go:226-232, core/knn.go:170-175)."""
    total, count = 0.0, 0.0
    for x in vals:
        total += float(x)
        count += 1.0
    mean = total / count if count else math.nan
    sq = 0.0
    for x in vals:
        sq += (float(x) - mean) * (float(x) - mean)
    std = math.sqrt(sq / count) + 1e-5 if count else math.nan
    return mean, std


def user_lists(u, i, r, users=None):
    """Each user's ratings as a list of inner item ids in dataset order: (user inner ids, ptr, ids, vals).  users:
    the inner user ids to take (default all, ascending)."""
    iu, ii = inner_of(np.asarray(u)), inner_of(np.asarray(i))
    r = np.asarray(r, dtype=np.float64)
    users = np.arange(int(iu.max()) + 1) if users is None else np.asarray(users)
    ptr, ids, vals = [0], [], []
    for q in users.tolist():
        sel = np.flatnonzero(iu == q)
        ids.append(ii[sel])
        vals.append(r[sel])
        ptr.append(ptr[-1] + len(sel))
    return users, np.array(ptr, dtype=np.int64), np.concatenate(ids), np.concatenate(vals)


def lists_of_raw(u_train, i_train, u, i, r):
    """Ratings (u, i, r) of users of the train set as lists over the train set's inner ids, one list per train
    user in inner order (users without a rating here get an empty list), items the train set does not know dropped:
    (ptr, ids, vals)."""
    users, items = raw_by_inner(np.asarray(u_train)), raw_by_inner(np.asarray(i_train))
    uix = {v: n for n, v in enumerate(users.tolist())}
    iix = {v: n for n, v in enumerate(items.tolist())}
    lists = [[] for _ in users]
    for uu, it, rr in zip(np.asarray(u).tolist(), np.asarray(i).tolist(), np.asarray(r, dtype=np.float64).tolist()):
        if uu in uix and it in iix:
            lists[uix[uu]].append((iix[it], rr))
    ptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
    ids = np.array([a for x in lists for a, _ in x], dtype=np.int64)
    vals = np.array([b for x in lists for _, b in x], dtype=np.float64)
    return ptr, ids, vals
