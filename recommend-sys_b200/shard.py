"""Sharding of the similarity rows across the GPUs of one box (SURVEY.md §8e): one process per GPU,
torch.distributed (NCCL over NVLink; gloo in the CPU tests) is the plumbing, not the product.

Three schemes, all with the rating matrix replicated on every GPU (it replaces the goroutine row
split of core/knn.go:192-216):
  * contiguous row shards (`shard_rows`): a rank computes full rows [begin, end) against all N rows
    (tensor path: 128-aligned) and all-gathers neighbour lists / predictions;
  * symmetric slabs (top-k only, config 4): slabs dealt in snake order, every pair computed once,
    partial neighbour lists all-gathered and united;
  * CYCLIC ROW SHARDS (`ShardedKNN`, the strong-scaling form of Fit + Predict): rows dealt in blocks
    of 32, every pair computed once by the exact sparse kernel, the other triangle of a rank's rows
    pulled from the peers' matrices over NVLink (rs_knn_mirror, CUDA IPC), the test pairs routed to
    the owner of their left row, predictions all-gathered."""
from __future__ import annotations


def shard_rows(n: int, world: int, rank: int, align: int = 128):
    """[begin,end) of the left rows owned by `rank`: contiguous, `align`-row aligned boundaries
    (the tensor-core tile height) except for the last shard, sizes differing by <= align."""
    blocks = (n + align - 1) // align
    b0 = blocks * rank // world
    b1 = blocks * (rank + 1) // world
    return min(b0 * align, n), min(b1 * align, n)


def allgather_topk(idx_local, sim_local, n: int, k: int, group=None, align: int = 128):
    """All-gather the per-shard neighbour lists into the full (n, k) lists on every rank.
    idx_local/sim_local: torch tensors (rows_of_this_rank, k) on the collective's device."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    bounds = [shard_rows(n, world, r, align) for r in range(world)]
    max_rows = max(b - a for a, b in bounds)
    pad_i = torch.full((max_rows, k), -1, dtype=torch.int32, device=idx_local.device)
    pad_s = torch.full((max_rows, k), float("nan"), dtype=torch.float64, device=sim_local.device)
    pad_i[: idx_local.shape[0]] = idx_local
    pad_s[: sim_local.shape[0]] = sim_local
    all_i = torch.empty((world * max_rows, k), dtype=torch.int32, device=idx_local.device)
    all_s = torch.empty((world * max_rows, k), dtype=torch.float64, device=sim_local.device)
    dist.all_gather_into_tensor(all_i, pad_i, group=group)
    dist.all_gather_into_tensor(all_s, pad_s, group=group)
    out_i = torch.cat([all_i[r * max_rows: r * max_rows + (b - a)] for r, (a, b) in enumerate(bounds)])
    out_s = torch.cat([all_s[r * max_rows: r * max_rows + (b - a)] for r, (a, b) in enumerate(bounds)])
    return out_i, out_s


def slab_owner(slab: int, world: int) -> int:
    """Which shard computes slab `slab` under symmetric-slab sharding: slabs are dealt in snake order
    (0..world-1, world-1..0, ...) because slab s costs ~ (n_slabs - s) — the same rule as csrc/topk.cu."""
    rnd, pos = divmod(slab, world)
    return world - 1 - pos if rnd & 1 else pos


def allgather_partial_topk(idx_part, sim_part, group=None):
    """Symmetric-slab sharding (rs_knn_params.shard_count >= 1): every rank holds PARTIAL neighbour
    lists for all n rows, (n, k).  Returns the stacked (world, n, k) tensors on every rank — the one
    exchange step of the sharded Fit, an all-gather over NCCL/NVLink (gloo in the CPU tests)."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    n, k = idx_part.shape
    all_i = torch.empty((world * n, k), dtype=idx_part.dtype, device=idx_part.device)
    all_s = torch.empty((world * n, k), dtype=sim_part.dtype, device=sim_part.device)
    dist.all_gather_into_tensor(all_i, idx_part.contiguous(), group=group)
    dist.all_gather_into_tensor(all_s, sim_part.contiguous(), group=group)
    return all_i.view(world, n, k), all_s.view(world, n, k)


def union_topk_device(all_i, all_s):
    """Unites stacked partial lists (n_lists, n, k) into the final (n, k) lists on the device
    (rs_knn_topk_union_device; CUDA tensors, the current torch stream)."""
    import torch

    from . import core

    n_lists, n, k = all_i.shape
    out_i = torch.empty((n, k), dtype=torch.int32, device=all_i.device)
    out_s = torch.empty((n, k), dtype=torch.float64, device=all_s.device)
    core._check(core.knn_lib().rs_knn_topk_union_device(
        n_lists, n, k, all_i.data_ptr(), all_s.data_ptr(), out_i.data_ptr(), out_s.data_ptr(),
        torch.cuda.current_stream(all_i.device).cuda_stream))
    return out_i, out_s


UNION_CAP = 2048   # entries rs_knn_topk_union_device unites per row: n_lists * k <= 2048


def union_recommend_device(all_i, all_s, unite=None):
    """Unites stacked partial top-N lists (n_lists, n, n_top) — one list per row shard, from
    rs_knn_recommend_sharded_device — into the final (n, n_top) lists.  A union call takes at most
    UNION_CAP // n_top lists; more are united in groups of that many and the results again, a tree of the
    same kernel (valid because every target is in at most one partial list).  `unite` replaces
    union_topk_device (tests)."""
    unite = unite or union_topk_device
    n_lists, n, n_top = all_i.shape
    if n == 0:
        return all_i[0], all_s[0]
    group = UNION_CAP // n_top
    while True:
        parts = [unite(all_i[g:g + group], all_s[g:g + group]) for g in range(0, n_lists, group)]
        if len(parts) == 1:
            return parts[0]
        all_i = all_i.new_empty((len(parts), n, n_top))
        all_s = all_s.new_empty((len(parts), n, n_top))
        for p, (pi, ps) in enumerate(parts):
            all_i[p], all_s[p] = pi, ps
        n_lists = len(parts)


def allgather_predictions(pred_local, counts, group=None):
    """All-gather per-rank prediction vectors of (known) lengths `counts` into one vector."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    m = max(counts)
    pad = torch.zeros(m, dtype=torch.float64, device=pred_local.device)
    pad[: pred_local.shape[0]] = pred_local
    out = torch.empty(world * m, dtype=torch.float64, device=pred_local.device)
    dist.all_gather_into_tensor(out, pad, group=group)
    return torch.cat([out[r * m: r * m + c] for r, c in enumerate(counts)])


# ---------------------------------------------------------------------------------------------
# Cyclic row shards: Fit + Predict of ONE matrix on all ranks (strong scaling)
# ---------------------------------------------------------------------------------------------
def route_pairs(left_inner, world):
    """Owner rank of every test pair: the shard that owns its left row (cyclic, blocks of 32); pairs
    with an unknown left id (cold start, answered with GlobalMean by any shard) are spread evenly."""
    import numpy as np

    from . import core

    left_inner = np.asarray(left_inner)
    owner = core.cyclic_owner(np.maximum(left_inner, 0), world)
    cold = left_inner < 0
    if cold.any():
        owner = owner.copy()
        owner[cold] = np.arange(int(cold.sum())) % world
    return owner


def attach_peers_and_mirror(handle, group=None):
    """The exchange step of a cyclic-sharded Fit.  Every rank waits for its own Fit, the 72-byte
    (CUDA IPC handle, offset) records are all-gathered — which is also the barrier that tells a rank
    every peer's triangle is complete — and the rank pulls the other triangle of its rows from the
    peers' matrices (rs_knn_mirror: P2P loads over NVLink)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    hb, off = handle.peer_export()
    rec = np.concatenate([hb, np.array([off], dtype=np.int64).view(np.uint8)])
    handle.synchronize()                      # own triangle complete before anybody is told so
    dev = torch.device("cuda", torch.cuda.current_device())
    mine = torch.from_numpy(rec).to(dev)
    allr = torch.empty(world * 72, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(allr, mine, group=group)
    allr = allr.cpu().numpy().reshape(world, 72)
    handle.peer_import(allr[:, :64].copy(), allr[:, 64:].copy().view(np.int64).reshape(world))
    handle.mirror()


class ShardedKNN:
    """KNN.Fit / DataSet.Predict of ONE training set on all ranks of the process group — the
    multi-GPU form of core/knn.go:143-217 + core/data.go:98-105.  Wraps a core.KNN:

        est = ShardedKNN(rs.NewKNNWithMean(params))      # same constructors, same Parameters
        est.Fit(train)                                   # every rank passes the same TrainSet
        preds = est.PredictBatch(users, items)           # full prediction vector on every rank
        est.Update(new_ratings)                          # every rank passes the same DataSet

    Fit uploads 1/world of the ratings per rank from (pinned) host memory and all-gathers them over
    NVLink, so the host->device traffic is divided by the number of GPUs."""

    def __init__(self, knn, group=None):
        import torch.distributed as dist

        self.knn = knn
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self._need_mirror = False
        self._split = False         # an Update succeeded on some ranks only: every call refuses until the next Fit

    def Fit(self, trainSet):
        import numpy as np
        import torch
        import torch.distributed as dist

        k = self.knn
        sim, left, right, n_left, n_right, lb, rbias, gb = k._prepare(trainSet)
        dev = torch.device("cuda", torch.cuda.current_device())
        nnz = len(left)
        per = (nnz + self.world - 1) // self.world
        lo, hi = min(nnz, self.rank * per), min(nnz, (self.rank + 1) * per)

        def gather(a, dtype):
            part = torch.zeros(per, dtype=dtype, device=dev)
            part[: hi - lo].copy_(torch.from_numpy(a[lo:hi]), non_blocking=True)     # H2D of this rank's slice only
            out = torch.empty(per * self.world, dtype=dtype, device=dev)
            dist.all_gather_into_tensor(out, part, group=self.group)
            return out

        d_left, d_right = gather(left, torch.int32), gather(right, torch.int32)
        d_rating = gather(trainSet.Ratings, torch.float64)
        d_lb = torch.from_numpy(np.ascontiguousarray(lb, dtype=np.float64)).to(dev) if lb is not None else None
        d_rb = torch.from_numpy(np.ascontiguousarray(rbias, dtype=np.float64)).to(dev) if rbias is not None else None
        k.Close()
        k._h = k._new_handle(sim, shard_count=self.world, shard_index=self.rank, device=dev.index)
        k._h.set_stream(torch.cuda.current_stream(dev).cuda_stream)
        k._h.fit_device(d_left.data_ptr(), d_right.data_ptr(), d_rating.data_ptr(), nnz, n_left, n_right,
                        trainSet.GlobalMean, d_lb.data_ptr() if d_lb is not None else 0,
                        d_rb.data_ptr() if d_rb is not None else 0, gb)
        self._keep = (d_left, d_right, d_rating, d_lb, d_rb)
        # like rs_knn_fit, Fit returns while the similarity kernel runs: the exchange step (which waits for
        # it, here and on every peer) is deferred to the first call that needs the whole rows, so the host
        # work in between — converting and routing the test set's ids — overlaps the kernel
        self._need_mirror = True
        self._split = False
        return self

    def _device(self):
        """This rank's GPU: the update's inputs and the all-reduce of its return codes."""
        import torch

        return torch.device("cuda", torch.cuda.current_device())

    def _refuse_if_split(self):
        if self._split:
            raise RuntimeError("ShardedKNN: an Update succeeded on some ranks and failed on others, so the shards no "
                               "longer hold one model; Fit again")

    def _finish_fit(self):
        self._refuse_if_split()
        if self._need_mirror:
            attach_peers_and_mirror(self.knn._h, self.group)
            self.knn._after_fit()
            self._need_mirror = False

    def PredictBatch(self, userIDs, itemIDs):
        import numpy as np
        import torch
        import torch.distributed as dist

        self._refuse_if_split()
        k = self.knn
        n = len(userIDs)
        if n == 0:
            self._finish_fit()
            return np.empty(0, dtype=np.float64)
        # Inner ids are written straight into pinned staging memory (torch's caching host allocator: no
        # cudaHostAlloc after the first call) by the threaded host conversion, which runs beside the similarity
        # kernel (Fit has returned, the kernel has not).  Every rank gets the FULL test set (32 MB at 4 M pairs —
        # cheaper than routing it on the host); a shard answers the pairs whose left row it owns and leaves +0.0
        # elsewhere; an int64 SUM all-reduce of the bit patterns over NVLink assembles the vector exactly
        # (x + 0 + ... + 0 in integer arithmetic).
        dev = torch.device("cuda", torch.cuda.current_device())
        p_l = torch.empty(n, dtype=torch.int32, pin_memory=True)
        p_r = torch.empty(n, dtype=torch.int32, pin_memory=True)
        k.Data.convert_users(userIDs, out=(p_l if k._userBased else p_r).numpy())
        k.Data.convert_items(itemIDs, out=(p_r if k._userBased else p_l).numpy())
        d_l = p_l.to(dev, non_blocking=True)
        d_r = p_r.to(dev, non_blocking=True)
        d_o = torch.empty(n, dtype=torch.float64, device=dev)
        self._finish_fit()
        k._h.predict_batch_sharded_device(d_l.data_ptr(), d_r.data_ptr(), n, d_o.data_ptr())
        dist.all_reduce(d_o.view(torch.int64), op=dist.ReduceOp.SUM, group=self.group)
        out = torch.empty(n, dtype=torch.float64, pin_memory=True)
        out.copy_(d_o, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return out.numpy()

    def Predict(self, userID, itemID):
        import numpy as np

        return float(self.PredictBatch(np.array([userID]), np.array([itemID]))[0])

    def Update(self, rowSet):
        """KNN.Update on the row shards: every rank passes the same `rowSet`, extends Data with it and adds it to its
        shard (rs_knn_update_sharded_device), with no exchange of data; afterwards every rank holds its rows of the Fit
        of Data.Extend(rowSet), bit for bit.  The ranks then agree on the outcome: a refusal (the same on every rank,
        since every check reads replicated data) raises on every rank and leaves the model as it was everywhere; an
        update that succeeded on some ranks and failed on others (out of memory, a CUDA error) raises on every rank,
        and every later call raises until the next Fit."""
        import numpy as np
        import torch
        import torch.distributed as dist

        from . import core

        self._finish_fit()
        k = self.knn
        data = k.Data.Extend(rowSet)
        n0 = k.Data.Length()
        iu, ii = data.innerUsers[n0:], data.innerItems[n0:]
        if k._userBased:
            left, right, n_left, n_right = iu, ii, data.UserCount, data.ItemCount
        else:
            left, right, n_left, n_right = ii, iu, data.ItemCount, data.UserCount
        dev = self._device()
        d_l = torch.from_numpy(np.ascontiguousarray(left, dtype=np.int32)).to(dev)
        d_r = torch.from_numpy(np.ascontiguousarray(right, dtype=np.int32)).to(dev)
        d_v = torch.from_numpy(np.ascontiguousarray(data.Ratings[n0:], dtype=np.float64)).to(dev)
        err = None
        try:
            k._h.update_sharded_device(d_l.data_ptr(), d_r.data_ptr(), d_v.data_ptr(), len(d_v), n_left, n_right,
                                       data.GlobalMean)
        except core.RsError as e:
            err = e
        code = err.code if err is not None else 0
        agree = torch.tensor([code, -code], dtype=torch.int64, device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN, group=self.group)
        lo, hi = int(agree[0]), -int(agree[1])
        if lo != hi:
            self._split = True
            raise core.RsError(lo, f"ShardedKNN.Update: the ranks disagree (return codes {lo} .. {hi}, this rank "
                                   f"{code}{': ' + str(err) if err is not None else ''}); every call refuses until "
                                   "the next Fit")
        if err is not None:
            raise err
        k.Data = data
        k.GlobalMean = data.GlobalMean
        k._after_fit()

    def _device_queries(self, userIDs):
        """The query side and the inner-id queries on this rank's GPU (every rank passes the same users)."""
        import numpy as np
        import torch

        self._finish_fit()
        side, q = self.knn._user_queries(userIDs)
        dev = torch.device("cuda", torch.cuda.current_device())
        return side, torch.from_numpy(np.ascontiguousarray(q, dtype=np.int32)).to(dev)

    def Recommend(self, userIDs, n):
        """KNN.Recommend on the row shards: each rank lists the best targets it can score (its own items for an
        item-based KNN, its own users' lists for a user-based one), the partial lists are all-gathered and
        united.  The same (items, scores) on every rank, bit for bit those of one unsharded KNN."""
        import numpy as np
        import torch

        side, d_q = self._device_queries(userIDs)
        m = d_q.shape[0]
        if m == 0:
            return np.empty((0, n), dtype=np.int64), np.empty((0, n), dtype=np.float64)
        ids = torch.empty((m, n), dtype=torch.int32, device=d_q.device)
        scores = torch.empty((m, n), dtype=torch.float64, device=d_q.device)
        self.knn._h.recommend_sharded_device(side, d_q.data_ptr(), m, n, ids.data_ptr(), scores.data_ptr())
        all_i, all_s = allgather_partial_topk(ids, scores, self.group)
        ui, us = union_recommend_device(all_i, all_s)
        return self.knn._raw_items(ui.cpu().numpy()), us.cpu().numpy()

    def ScoreAll(self, userIDs):
        """KNN.ScoreAll on the row shards: each rank scores the cells it owns, +0.0 elsewhere, and an int64 SUM
        all-reduce of the bit patterns assembles the rows, as PredictBatch does.  The full rows on every rank."""
        import torch
        import torch.distributed as dist

        from . import core

        side, d_q = self._device_queries(userIDs)
        m = d_q.shape[0]
        out = torch.empty((m, self.knn._h._n_targets(core.RS_SIDE[side])), dtype=torch.float64, device=d_q.device)
        if m:
            self.knn._h.score_all_sharded_device(side, d_q.data_ptr(), m, out.data_ptr())
            dist.all_reduce(out.view(torch.int64), op=dist.ReduceOp.SUM, group=self.group)
        return out.cpu().numpy()

    def ScoreAllGiven(self, dataSet):
        """KNN.ScoreAllGiven is not available on row shards yet (the library refuses them)."""
        raise NotImplementedError("ScoreAllGiven: row-sharded handles are not supported; use an unsharded KNN")

    def RecommendGiven(self, dataSet, n):
        """KNN.RecommendGiven is not available on row shards yet (the library refuses them)."""
        raise NotImplementedError("RecommendGiven: row-sharded handles are not supported; use an unsharded KNN")

    def Close(self):
        self.knn.Close()
