"""Host-side mirror of the reference's Go package `core` for the KNN hot path, in Python over
the C ABI (include/rs_knn.h) — the same names, argument meaning and error behaviour, so the
parity tests read like the reference's own tests.

    reference (Go)                                   here
    ---------------------------------------------    ------------------------------------------
    core/base.go:14-57   Parameters + typed getters   Parameters
    core/sim.go:7        type Sim / Cosine MSD Pearson Sim objects Cosine, MSD, Pearson (+PearsonBaseline ext.)
    core/data.go:21-105  DataSet, KFold, Predict       DataSet
    core/data.go:109-216 TrainSet, NewTrainSet         TrainSet / NewTrainSet
    core/knn.go:50-73    NewKNN, NewKNNWithMean, ...   same names
    core/knn.go:143-217  KNN.Fit                       KNN.Fit  -> rs_knn_fit
    core/knn.go:75-141   KNN.Predict                   KNN.Predict / KNN.PredictBatch -> rs_knn_predict_batch
    core/base.go:108-163 BaseLine                      BaseLine (host SGD, rs_host_baseline_sgd)
    core/eval.go:18-67   CrossValidate                 CrossValidate (intended 6-argument form, SURVEY.md §4.3)
    core/utils.go:160-180 RMSE / MAE                   RMSE / MAE on (predictions, truth)

The reference is Go; no Go toolchain exists in the build image, so this Python mirror is the
runnable host side (the cgo bridge a maintainer would add is in go/ and INTEGRATION.md).
There is NO CPU fallback: every Fit/Predict runs on the CUDA device through librs_knn_b200.so
and raises if the library or a device is missing.
"""
from __future__ import annotations

import ctypes as C
import os
import math
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
_LIB_KNN = Path(os.environ.get("RS_KNN_LIB", _PKG / "librs_knn_b200.so"))   # RS_KNN_LIB: an alternative build
_LIB_HOST = _PKG / "librs_host.so"

RS_OK = 0
newID = -1  # core/data.go:129

# enum values of include/rs_knn.h
RS_SIM = {"cosine": 0, "msd": 1, "pearson": 2, "pearson_baseline": 3, "slope_one": 4}
RS_KNN_TYPE = {"basic": 0, "centered": 1, "zscore": 2, "baseline": 3}
RS_PEARSON_MODE = {"exact": 0, "sums": 1}
RS_SIM_PATH = {"auto": 0, "tensor": 1, "stream": 2}
RS_STORE = {"matrix": 0, "topk": 1}
RS_SIDE = {"left": 0, "right": 1}

basic, centered, zScore, baseline = "basic", "centered", "zscore", "baseline"  # core/knn.go:10-15


class RsKnnParams(C.Structure):
    _fields_ = [("sim", C.c_int32), ("knn_type", C.c_int32), ("k", C.c_int32), ("min_k", C.c_int32),
                ("device", C.c_int32), ("pearson_mode", C.c_int32), ("sim_path", C.c_int32),
                ("store", C.c_int32), ("topk", C.c_int32), ("reserved0", C.c_int32),
                ("row_begin", C.c_int64), ("row_end", C.c_int64), ("shrinkage", C.c_double),
                ("shard_count", C.c_int32), ("shard_index", C.c_int32)]


class RsKnnProfile(C.Structure):
    _fields_ = [("sim_kernel_ms", C.c_double), ("predict_kernel_ms", C.c_double), ("prep_ms", C.c_double),
                ("sim_launches", C.c_int64), ("predict_launches", C.c_int64), ("total_launches", C.c_int64),
                ("sim_path_used", C.c_int32), ("reserved0", C.c_int32), ("corated_triples", C.c_double)]


ABI_SYMBOLS = [
    "rs_last_error", "rs_knn_abi_version", "rs_knn_device_count", "rs_knn_params_default", "rs_knn_create",
    "rs_knn_destroy", "rs_knn_set_stream", "rs_knn_fit", "rs_knn_fit_device", "rs_knn_predict_batch",
    "rs_knn_predict_batch_device", "rs_knn_predict_neighbors", "rs_knn_sims_rows", "rs_knn_topk",
    "rs_knn_topk_device", "rs_knn_cosums", "rs_knn_means", "rs_knn_stddevs", "rs_knn_profile_get",
    "rs_knn_profile_reset", "rs_knn_synchronize", "rs_knn_trim_cache", "rs_baseline_als",
    "rs_knn_topk_union_device", "rs_knn_set_k", "rs_knn_peer_export", "rs_knn_peer_import",
    "rs_knn_peer_import_local", "rs_knn_mirror", "rs_knn_predict_batch_sharded_device", "rs_knn_host_alloc",
    "rs_knn_host_free", "rs_knn_score_all", "rs_knn_score_all_device", "rs_knn_recommend", "rs_knn_recommend_device",
    "rs_knn_score_all_sharded_device", "rs_knn_recommend_sharded_device", "rs_knn_score_all_given",
    "rs_knn_score_all_given_device", "rs_knn_recommend_given", "rs_knn_recommend_given_device", "rs_knn_update",
    "rs_knn_update_device",
]

_knn_lib = None
_host_lib = None


def knn_lib():
    """librs_knn_b200.so with argtypes set.  Raises if the extension was not built."""
    global _knn_lib
    if _knn_lib is not None:
        return _knn_lib
    if not _LIB_KNN.exists():
        raise RuntimeError(f"{_LIB_KNN} is missing: build the CUDA extension first "
                           "(python -c 'import __graft_entry__ as g; g.build()'); there is no CPU fallback")
    L = C.CDLL(str(_LIB_KNN))
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    L.rs_last_error.restype = C.c_char_p
    L.rs_knn_abi_version.restype = i32
    L.rs_knn_device_count.restype = i32
    L.rs_knn_params_default.argtypes = [C.POINTER(RsKnnParams)]
    L.rs_knn_create.argtypes = [C.POINTER(RsKnnParams), C.POINTER(vp)]
    L.rs_knn_destroy.argtypes = [vp]
    L.rs_knn_set_stream.argtypes = [vp, vp, i32]
    L.rs_knn_fit.argtypes = [vp, vp, vp, vp, i64, i32, i32, dbl, vp, vp, dbl]
    L.rs_knn_fit_device.argtypes = [vp, vp, vp, vp, i64, i32, i32, dbl, vp, vp, dbl]
    L.rs_knn_predict_batch.argtypes = [vp, vp, vp, i64, vp]
    L.rs_knn_predict_batch_device.argtypes = [vp, vp, vp, i64, vp]
    L.rs_knn_predict_neighbors.argtypes = [vp, i32, i32, i32, vp, vp, C.POINTER(i32)]
    L.rs_knn_sims_rows.argtypes = [vp, i64, i64, vp]
    L.rs_knn_topk.argtypes = [vp, i32, vp, vp]
    L.rs_knn_topk_device.argtypes = [vp, i32, vp, vp]
    L.rs_knn_cosums.argtypes = [vp, i64, i64, vp]
    L.rs_knn_means.argtypes = [vp, vp]
    L.rs_knn_stddevs.argtypes = [vp, vp]
    L.rs_knn_profile_get.argtypes = [vp, C.POINTER(RsKnnProfile)]
    L.rs_knn_profile_reset.argtypes = [vp]
    L.rs_knn_synchronize.argtypes = [vp]
    for name in ABI_SYMBOLS:
        if name != "rs_last_error":
            getattr(L, name).restype = i32
    L.rs_baseline_als.argtypes = [i32, vp, vp, vp, i64, i32, i32, dbl, dbl, dbl, i32, vp, vp]
    L.rs_knn_topk_union_device.argtypes = [i32, i64, i32, vp, vp, vp, vp, vp]
    L.rs_knn_set_k.argtypes = [vp, i32, i32]
    L.rs_knn_peer_export.argtypes = [vp, vp, C.POINTER(i64)]
    L.rs_knn_peer_import.argtypes = [vp, i32, vp, vp]
    L.rs_knn_peer_import_local.argtypes = [vp, i32, vp]
    L.rs_knn_mirror.argtypes = [vp]
    L.rs_knn_predict_batch_sharded_device.argtypes = [vp, vp, vp, i64, vp]
    L.rs_knn_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.rs_knn_host_free.argtypes = [vp]
    L.rs_knn_score_all.argtypes = [vp, i32, vp, i64, vp]
    L.rs_knn_score_all_device.argtypes = [vp, i32, vp, i64, vp]
    L.rs_knn_recommend.argtypes = [vp, i32, vp, i64, i32, vp, vp]
    L.rs_knn_recommend_device.argtypes = [vp, i32, vp, i64, i32, vp, vp]
    L.rs_knn_score_all_sharded_device.argtypes = [vp, i32, vp, i64, vp]
    L.rs_knn_recommend_sharded_device.argtypes = [vp, i32, vp, i64, i32, vp, vp]
    L.rs_knn_score_all_given.argtypes = [vp, i32, vp, vp, vp, i64, vp]
    L.rs_knn_score_all_given_device.argtypes = [vp, i32, vp, vp, vp, i64, vp]
    L.rs_knn_recommend_given.argtypes = [vp, i32, vp, vp, vp, i64, i32, vp, vp]
    L.rs_knn_recommend_given_device.argtypes = [vp, i32, vp, vp, vp, i64, i32, vp, vp]
    L.rs_knn_update.argtypes = [vp, vp, vp, vp, i64, i32, i32, dbl]
    L.rs_knn_update_device.argtypes = [vp, vp, vp, vp, i64, i32, i32, dbl]
    _knn_lib = L
    return L


def host_lib():
    global _host_lib
    if _host_lib is not None:
        return _host_lib
    if not _LIB_HOST.exists():
        raise RuntimeError(f"{_LIB_HOST} is missing: run __graft_entry__.build()")
    L = C.CDLL(str(_LIB_HOST))
    L.rs_host_inner_ids.restype = C.c_int64
    L.rs_host_inner_ids.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.rs_host_baseline_sgd.restype = None
    L.rs_host_baseline_sgd.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                       C.c_double, C.c_double, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.POINTER(C.c_double)]
    L.rs_host_synth_ratings.restype = C.c_int64
    L.rs_host_synth_ratings.argtypes = [C.c_int32, C.c_int32, C.c_int64, C.c_uint64, C.c_void_p, C.c_void_p,
                                        C.c_void_p]
    L.rs_host_mean_seq.restype = C.c_double
    L.rs_host_mean_seq.argtypes = [C.c_void_p, C.c_int64]
    L.rs_host_save_neighbors.restype = C.c_int32
    L.rs_host_save_neighbors.argtypes = [C.c_char_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    L.rs_host_load_neighbors.restype = C.c_int32
    L.rs_host_load_neighbors.argtypes = [C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.c_void_p,
                                         C.c_void_p]
    L.rs_host_load_ratings.restype = C.c_int64
    L.rs_host_load_ratings.argtypes = [C.c_char_p, C.c_char_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_int64]
    L.rs_host_route_pairs.restype = None
    L.rs_host_route_pairs.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.rs_host_convert_dense.restype = None
    L.rs_host_convert_dense.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    L.rs_host_convert_dense_mt.restype = None
    L.rs_host_convert_dense_mt.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32]
    _host_lib = L
    return L


class RsError(RuntimeError):
    """Non-zero status from the C ABI.  The Go wrapper panics here (the reference's own
    convention on this path: core/base.go:68-74, type-assertion panics core/base.go:26-54)."""

    def __init__(self, code, msg):
        super().__init__(f"rs_knn error {code}: {msg}")
        self.code = code


def _check(rc):
    if rc != RS_OK:
        raise RsError(rc, knn_lib().rs_last_error().decode("utf-8", "replace"))


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# --------------------------------------------------------------------------------------------
# core/sim.go:7 — `type Sim func(SortedIdRatings, SortedIdRatings) float64`
# --------------------------------------------------------------------------------------------
class SortedIdRatings:
    """core/data.go:245-265; NewSortedIdRatings sorts by id (core/data.go:249-253)."""

    def __init__(self, pairs):
        self.data = sorted(((int(i), float(r)) for i, r in pairs), key=lambda t: t[0])

    def Len(self):
        return len(self.data)


def NewSortedIdRatings(pairs):
    return SortedIdRatings(pairs)


class Sim:
    """A similarity of the reference as a first-class value (Parameters["sim"], core/base.go:45-50).
    Calling it on two SortedIdRatings evaluates that one pair ON THE DEVICE (a 2-row Fit), which
    is how the reference's own known-answer tests (core/sim_test.go) are replayed here."""

    def __init__(self, name):
        self.name = name

    def __repr__(self):
        return f"Sim({self.name})"

    def __call__(self, a: SortedIdRatings, b: SortedIdRatings, **device_opts) -> float:
        ids = sorted({i for i, _ in a.data} | {i for i, _ in b.data})
        col = {v: x for x, v in enumerate(ids)}
        left = np.array([0] * len(a.data) + [1] * len(b.data), dtype=np.int32)
        right = np.array([col[i] for i, _ in a.data] + [col[i] for i, _ in b.data], dtype=np.int32)
        rating = np.array([r for _, r in a.data] + [r for _, r in b.data], dtype=np.float64)
        if len(a.data) == 0 or len(b.data) == 0:
            return math.nan  # 0/0 in every core/sim.go formula
        h = _Handle(sim=self.name, **device_opts)
        try:
            h.fit(left, right, rating, 2, max(1, len(ids)), float(rating.mean()))
            return float(h.sims_rows(0, 1)[0, 1])
        finally:
            h.close()


Cosine = Sim("cosine")            # core/sim.go:10
MSD = Sim("msd")                  # core/sim.go:28
Pearson = Sim("pearson")          # core/sim.go:47
PearsonBaseline = Sim("pearson_baseline")  # extension (north star), not in the reference
_SIMS_BY_NAME = {s_.name: s_ for s_ in (Cosine, MSD, Pearson, PearsonBaseline)}


# --------------------------------------------------------------------------------------------
# core/base.go:14-57 — Parameters
# --------------------------------------------------------------------------------------------
class Parameters(dict):
    def Copy(self):
        return Parameters(self)

    def _get(self, name, default, typ, what):
        if name in self:
            val = self[name]
            if typ is float and isinstance(val, int) and not isinstance(val, bool):
                raise TypeError(f"interface conversion: Parameters[{name!r}] is int, not float64")
            if not isinstance(val, typ) or (typ is int and isinstance(val, bool)):
                # Go: val.(T) panics on a wrong dynamic type (core/base.go:26-54)
                raise TypeError(f"interface conversion: Parameters[{name!r}] is {type(val).__name__}, not {what}")
            return val
        return default

    def GetInt(self, name, _default):
        return self._get(name, _default, int, "int")

    def GetBool(self, name, _default):
        return self._get(name, _default, bool, "bool")

    def GetFloat64(self, name, _default):
        return self._get(name, _default, float, "float64")

    def GetSim(self, name, _default):
        return self._get(name, _default, Sim, "core.Sim")

    def GetString(self, name, _default):
        return self._get(name, _default, str, "string")


def _params(p):
    return Parameters() if p is None else (p if isinstance(p, Parameters) else Parameters(p))


# --------------------------------------------------------------------------------------------
# core/data.go — DataSet / TrainSet
# --------------------------------------------------------------------------------------------
class DataSet:
    """core/data.go:21-105"""

    def __init__(self, users, items, ratings):
        self.Users = np.ascontiguousarray(users, dtype=np.int64)
        self.Items = np.ascontiguousarray(items, dtype=np.int64)
        self.Ratings = np.ascontiguousarray(ratings, dtype=np.float64)

    def Length(self):
        return len(self.Ratings)

    def Index(self, i):
        return int(self.Users[i]), int(self.Items[i]), float(self.Ratings[i])

    def SubSet(self, indices):
        return DataSet(self.Users[indices], self.Items[indices], self.Ratings[indices])

    def KFold(self, k, seed):
        """core/data.go:49-70.  The reference builds a seeded RNG and throws it away, so its folds
        are unreproducible (SURVEY.md hazard 3); here the permutation is numpy's for `seed`."""
        n = self.Length()
        perm = np.random.RandomState(seed & 0xFFFFFFFF).permutation(n)
        train_folds, test_folds = [], []
        fold_size = n // k
        begin = end = 0
        for i in range(k):
            end += fold_size
            if i < n % k:
                end += 1
            test_folds.append(self.SubSet(perm[begin:end]))
            train_folds.append(NewTrainSet(self.SubSet(np.concatenate([perm[:begin], perm[end:]]))))
            begin = end
        return train_folds, test_folds

    def Split(self, testSize, seed):
        """core/data.go:72-79"""
        n = self.Length()
        perm = np.random.RandomState(seed & 0xFFFFFFFF).permutation(n)
        mid = int(float(n) * testSize)
        return NewTrainSet(self.SubSet(perm[mid:])), self.SubSet(perm[:mid])

    def Predict(self, estimator):
        """core/data.go:98-105.  The reference loops Predict(u,i) serially; an estimator that
        implements the optional BatchPredictor interface (PredictBatch) gets the whole test set
        in one call — one cgo crossing, one kernel launch."""
        if hasattr(estimator, "PredictBatch"):
            return estimator.PredictBatch(self.Users, self.Items)
        return np.array([estimator.Predict(int(u), int(i)) for u, i in zip(self.Users, self.Items)])


def NewRawSet(users, items, ratings):
    return DataSet(users, items, ratings)


def _inner_ids(raw):
    inner = np.empty(len(raw), dtype=np.int32)
    count = host_lib().rs_host_inner_ids(_ptr(raw), len(raw), _ptr(inner))
    return inner, int(count)


def _global_mean(ratings):
    """core/data.go:134.  Integer ratings: the sum is exact in any order (vectorised); otherwise the
    sequential sum of the restatement (gonum's own order is pinned by no reference test)."""
    n = len(ratings)
    if n == 0:
        return math.nan
    r = np.ascontiguousarray(ratings, dtype=np.float64)
    if np.array_equal(r, np.rint(r)) and float(np.abs(r).max()) * n < 2.0 ** 53:
        return float(np.add.reduce(r) / n)
    return float(host_lib().rs_host_mean_seq(_ptr(r), n))


class TrainSet(DataSet):
    """core/data.go:109-216"""

    def __init__(self, rowSet: DataSet):
        super().__init__(rowSet.Users, rowSet.Items, rowSet.Ratings)
        # core/data.go:134 — stat.Mean(Ratings, nil)
        self.GlobalMean = _global_mean(self.Ratings)
        # core/data.go:137-151 — inner id = order of first appearance
        self.innerUsers, self.UserCount = _inner_ids(self.Users)
        self.innerItems, self.ItemCount = _inner_ids(self.Items)
        self._umap = None
        self._imap = None
        self._ulook = None
        self._ilook = None

    def _maps(self):
        if self._umap is None:
            self._umap = dict(zip(self.Users.tolist(), self.innerUsers.tolist()))
            self._imap = dict(zip(self.Items.tolist(), self.innerItems.tolist()))

    def ConvertUserID(self, userID):
        self._maps()
        return self._umap.get(int(userID), newID)

    def ConvertItemID(self, itemID):
        self._maps()
        return self._imap.get(int(itemID), newID)

    def convert_users(self, raw, out=None):
        """Vectorised ConvertUserID for a batch (newID = -1 for unseen ids)."""
        if self._ulook is None:
            self._ulook = _lookup_table(self.Users, self.innerUsers)
        return _convert(self._ulook, raw, out)

    def convert_items(self, raw, out=None):
        if self._ilook is None:
            self._ilook = _lookup_table(self.Items, self.innerItems)
        return _convert(self._ilook, raw, out)

    def RatingRange(self):
        return float(self.Ratings.min()), float(self.Ratings.max())

    def Extend(self, rowSet: DataSet) -> "TrainSet":
        """The TrainSet of this one's rows followed by `rowSet`'s: NewTrainSet of the concatenation, so the inner ids
        continue the order of first appearance (known ids keep theirs, new ones come after) and GlobalMean is that
        TrainSet's, bit for bit."""
        return TrainSet(DataSet(np.concatenate([self.Users, rowSet.Users]), np.concatenate([self.Items, rowSet.Items]),
                                np.concatenate([self.Ratings, rowSet.Ratings])))


class _HostBlock:
    """A page-locked host block of rs_knn_host_alloc; goes back to the library's cache with the last array on it."""

    def __init__(self, nbytes):
        p = C.c_void_p()
        _check(knn_lib().rs_knn_host_alloc(max(1, nbytes), C.byref(p)))
        self.ptr = p.value

    def __del__(self):
        try:
            knn_lib().rs_knn_host_free(self.ptr)
        except Exception:      # interpreter shutdown
            pass


def pinned_empty(n, dtype):
    """An uninitialised numpy array of n elements in page-locked host memory (full-speed, asynchronous copies to and
    from the device); ordinary memory if no CUDA device can provide it."""
    dtype = np.dtype(dtype)
    nbytes = int(n) * dtype.itemsize
    if nbytes == 0:
        return np.empty(0, dtype=dtype)
    try:
        blk = _HostBlock(nbytes)
    except (RsError, RuntimeError):
        return np.empty(n, dtype=dtype)
    buf = (C.c_char * nbytes).from_address(blk.ptr)
    buf._blk = blk                      # the array's base keeps the block alive
    return np.frombuffer(buf, dtype=dtype, count=int(n))


def _lookup_table(known_raw, known_inner):
    """raw id -> inner id.  Dense array when the raw ids are small non-negative integers (the
    usual case: MovieLens / Netflix ids), sorted table + binary search otherwise."""
    lo, hi = int(known_raw.min()), int(known_raw.max())
    if lo >= 0 and hi <= 8 * len(known_raw) + 1024:
        dense = np.full(hi + 2, newID, dtype=np.int32)
        dense[known_raw] = known_inner
        return ("dense", dense)
    uniq, first = np.unique(known_raw, return_index=True)
    return ("sorted", uniq, np.ascontiguousarray(known_inner[first]))


def host_threads():
    """Host threads one process may use for the id conversion: its share of the cores when several ranks
    (one per GPU) run on the box."""
    world = int(os.environ.get("LOCAL_WORLD_SIZE") or os.environ.get("WORLD_SIZE") or 1)
    return max(1, min(8, (os.cpu_count() or 1) // max(1, world)))


def _convert(table, raw, out=None):
    """Inner ids of `raw` (newID where unknown).  `out`: an int32 array to fill (e.g. pinned staging memory)."""
    raw = np.ascontiguousarray(raw, dtype=np.int64)
    if out is None:
        out = np.empty(len(raw), dtype=np.int32)
    assert out.dtype == np.int32 and out.flags.c_contiguous and len(out) == len(raw)
    if table[0] == "dense":
        dense = table[1]
        host_lib().rs_host_convert_dense_mt(_ptr(dense), len(dense) - 1, _ptr(raw), len(raw), _ptr(out), host_threads())
        return out
    _, uniq, inner = table
    pos = np.clip(np.searchsorted(uniq, raw), 0, len(uniq) - 1)
    out[:] = np.where(uniq[pos] == raw, inner[pos], newID)
    return out


def NewTrainSet(rowSet: DataSet) -> TrainSet:
    return TrainSet(rowSet)


def LoadDataFromFile(fileName, sep="\t", floatRatings=False, hasHeader=False):
    """core/data.go:287-310.  With the defaults this IS the reference's loader: fields 0..2 through
    strconv.Atoi, so half-star ratings ("3.5") and header lines silently become 0.  floatRatings=True
    (SURVEY.md §8 f-4) keeps fractional ratings — the device path fits any float64 rating —, hasHeader
    drops the first line (MovieLens-20M's ratings.csv has both).  Parsed by librs_host.so."""
    L = host_lib()
    path, bsep = os.fsencode(fileName), sep.encode()
    n = L.rs_host_load_ratings(path, bsep, int(floatRatings), int(hasHeader), None, None, None, 0)
    if n < 0:
        raise OSError(f"cannot read {fileName}")          # the reference log.Fatal()s here (core/data.go:294)
    users = np.empty(n, dtype=np.int64)
    items = np.empty(n, dtype=np.int64)
    ratings = np.empty(n, dtype=np.float64)
    L.rs_host_load_ratings(path, bsep, int(floatRatings), int(hasHeader), _ptr(users), _ptr(items), _ptr(ratings), n)
    return NewRawSet(users, items, ratings)


# --------------------------------------------------------------------------------------------
# core/dump.go — persistence (SURVEY.md §8 f-4)
# --------------------------------------------------------------------------------------------
def SaveNeighbors(fileName, idx, sim):
    """Neighbour lists (int32 idx, float64 sim)[n_rows][k] -> one checksummed binary file (rs_host.h)."""
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    sim = np.ascontiguousarray(sim, dtype=np.float64)
    if idx.ndim != 2 or idx.shape != sim.shape:
        raise ValueError("idx and sim must be (n_rows, k) arrays of the same shape")
    d = os.path.dirname(os.fspath(fileName))
    if d:
        os.makedirs(d, exist_ok=True)                     # core/dump.go:25 MkdirAll
    rc = host_lib().rs_host_save_neighbors(os.fsencode(fileName), idx.shape[0], idx.shape[1], _ptr(idx), _ptr(sim))
    if rc != 0:
        raise OSError(f"cannot write {fileName}")


def LoadNeighbors(fileName):
    L = host_lib()
    n, k = C.c_int64(0), C.c_int32(0)
    rc = L.rs_host_load_neighbors(os.fsencode(fileName), C.byref(n), C.byref(k), None, None)
    if rc == -1:
        raise OSError(f"cannot read {fileName}")
    if rc != 0:
        raise ValueError(f"{fileName} is not a neighbour-list file")
    idx = np.empty((n.value, k.value), dtype=np.int32)
    sim = np.empty((n.value, k.value), dtype=np.float64)
    rc = L.rs_host_load_neighbors(os.fsencode(fileName), C.byref(n), C.byref(k), _ptr(idx), _ptr(sim))
    if rc != 0:
        raise ValueError(f"{fileName}: truncated file or checksum mismatch")
    return idx, sim


def Save(fileName, estimator):
    """core/dump.go:23-36 for the estimators of this path.  gob writes the exported fields — for a KNN
    that includes the N x N Sims (5.7 GB at the MovieLens-20M shape).  Here the record is what is needed
    to REBUILD the estimator bit for bit: constructor, Parameters and the training triples in dataset
    order; Load refits on the device (76 ms at that shape — less than reading the matrix back)."""
    import json

    d = os.path.dirname(os.fspath(fileName))
    if d:
        os.makedirs(d, exist_ok=True)
    params = {}
    for key, val in (estimator.Params or {}).items():
        params[key] = {"__sim__": val.name} if isinstance(val, Sim) else val
    kind = "slope_one" if isinstance(estimator, SlopeOne) else "knn"
    meta = {"kind": kind, "knn_type": getattr(estimator, "KNNType", ""), "params": params,
            "fitted": estimator.Data is not None}
    ts = estimator.Data
    with open(fileName, "wb") as f:
        np.savez(f, meta=np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8),
                 users=ts.Users if ts is not None else np.empty(0, np.int64),
                 items=ts.Items if ts is not None else np.empty(0, np.int64),
                 ratings=ts.Ratings if ts is not None else np.empty(0, np.float64))


def Load(fileName):
    """core/dump.go:11-20: returns the estimator Save wrote, fitted (on the device) if it was."""
    import json

    with np.load(fileName, allow_pickle=False) as z:
        meta = json.loads(bytes(z["meta"]).decode())
        users, items, ratings = z["users"], z["items"], z["ratings"]
    params = Parameters()
    for key, val in meta["params"].items():
        params[key] = _SIMS_BY_NAME[val["__sim__"]] if isinstance(val, dict) and "__sim__" in val else val
    est = NewSlopeOne(params) if meta["kind"] == "slope_one" else KNN(meta["knn_type"], params)
    if meta["fitted"]:
        est.Fit(NewTrainSet(NewRawSet(users, items, ratings)))
    return est


CYC_B = 32   # RS_CYC_B of csrc/common.cuh: rows are dealt to cyclic shards in blocks of 32


def cyclic_rows(n, count, index):
    """Global ids of the rows shard `index` of `count` owns under cyclic row sharding."""
    i = np.arange(n)
    return i[(i // CYC_B) % count == index]


def cyclic_owner(ids, count):
    return (np.asarray(ids) // CYC_B) % count


def route_pairs_grouped(left_inner, count):
    """(order, counts): the test pairs grouped by the cyclic shard that owns their left row (stable; unknown
    left ids round-robin) — one counting-sort pass in librs_host.so."""
    left_inner = np.ascontiguousarray(left_inner, dtype=np.int32)
    order = np.empty(len(left_inner), dtype=np.int64)
    counts = np.zeros(count, dtype=np.int64)
    host_lib().rs_host_route_pairs(_ptr(left_inner), len(left_inner), count, CYC_B, _ptr(order), _ptr(counts))
    return order, counts.tolist()


# --------------------------------------------------------------------------------------------
# device handle
# --------------------------------------------------------------------------------------------
class _Handle:
    """Thin RAII wrapper of rs_knn* (in Go: an unexported field + Close()/finalizer)."""

    def __init__(self, sim="msd", knn_type="basic", k=40, min_k=1, device=-1, pearson_mode="exact",
                 sim_path="auto", store="matrix", topk=0, row_begin=0, row_end=0, shrinkage=0.0,
                 shard_count=0, shard_index=0):
        L = knn_lib()
        p = RsKnnParams()
        _check(L.rs_knn_params_default(C.byref(p)))
        p.sim, p.knn_type, p.k, p.min_k, p.device = RS_SIM[sim], RS_KNN_TYPE[knn_type], k, min_k, device
        p.pearson_mode, p.sim_path, p.store = RS_PEARSON_MODE[pearson_mode], RS_SIM_PATH[sim_path], RS_STORE[store]
        p.topk, p.row_begin, p.row_end, p.shrinkage = topk or k, row_begin, row_end, shrinkage
        p.shard_count, p.shard_index = shard_count, shard_index
        self.params = p
        self.h = C.c_void_p()
        _check(L.rs_knn_create(C.byref(p), C.byref(self.h)))
        self.n_left = self.n_right = 0
        self.rows = (0, 0)

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            knn_lib().rs_knn_destroy(self.h)
            self.h = None

    __del__ = close

    def set_stream(self, stream_ptr, use_own=False):
        """stream_ptr: a cudaStream_t as an int (0 = the legacy default stream)."""
        _check(knn_lib().rs_knn_set_stream(self.h, C.c_void_p(stream_ptr), int(use_own)))

    def fit(self, left, right, rating, n_left, n_right, global_mean, left_bias=None, right_bias=None,
            global_bias=0.0):
        left = np.ascontiguousarray(left, dtype=np.int32)
        right = np.ascontiguousarray(right, dtype=np.int32)
        rating = np.ascontiguousarray(rating, dtype=np.float64)
        lb = None if left_bias is None else np.ascontiguousarray(left_bias, dtype=np.float64)
        rb = None if right_bias is None else np.ascontiguousarray(right_bias, dtype=np.float64)
        _check(knn_lib().rs_knn_fit(self.h, _ptr(left), _ptr(right), _ptr(rating), len(rating), n_left, n_right,
                                    global_mean, None if lb is None else _ptr(lb),
                                    None if rb is None else _ptr(rb), global_bias))
        self._after_fit(n_left, n_right)

    def _after_fit(self, n_left, n_right):
        self.n_left, self.n_right = n_left, n_right
        rb, re = self.params.row_begin, self.params.row_end
        self.rows = (0, n_left) if (rb == 0 and re == 0) else (rb, re)

    def fit_device(self, d_left, d_right, d_rating, nnz, n_left, n_right, global_mean, d_left_bias=0,
                   d_right_bias=0, global_bias=0.0):
        """Arguments are raw device pointers (ints), e.g. torch tensors' data_ptr()."""
        _check(knn_lib().rs_knn_fit_device(self.h, d_left, d_right, d_rating, nnz, n_left, n_right, global_mean,
                                           d_left_bias or None, d_right_bias or None, global_bias))
        self._after_fit(n_left, n_right)

    def update(self, left, right, rating, n_left, n_right, global_mean):
        """Adds ratings to the fitted model: it becomes the Fit of the union, bit for bit (rs_knn_update)."""
        left = np.ascontiguousarray(left, dtype=np.int32)
        right = np.ascontiguousarray(right, dtype=np.int32)
        rating = np.ascontiguousarray(rating, dtype=np.float64)
        _check(knn_lib().rs_knn_update(self.h, _ptr(left), _ptr(right), _ptr(rating), len(rating), n_left, n_right,
                                       global_mean))
        self._after_fit(n_left, n_right)

    def update_device(self, d_left, d_right, d_rating, nnz, n_left, n_right, global_mean):
        _check(knn_lib().rs_knn_update_device(self.h, d_left, d_right, d_rating, nnz, n_left, n_right, global_mean))
        self._after_fit(n_left, n_right)

    def predict_batch(self, left, right):
        left = np.ascontiguousarray(left, dtype=np.int32)
        right = np.ascontiguousarray(right, dtype=np.int32)
        out = pinned_empty(len(left), np.float64) if len(left) >= 1 << 16 else np.empty(len(left), dtype=np.float64)
        _check(knn_lib().rs_knn_predict_batch(self.h, _ptr(left), _ptr(right), len(left), _ptr(out)))
        return out

    def predict_batch_device(self, d_left, d_right, n, d_out):
        _check(knn_lib().rs_knn_predict_batch_device(self.h, d_left, d_right, n, d_out))

    def predict_batch_sharded_device(self, d_left, d_right, n, d_out):
        _check(knn_lib().rs_knn_predict_batch_sharded_device(self.h, d_left, d_right, n, d_out))

    def predict_neighbors(self, left, right, cap=1024):
        ids = np.empty(cap, dtype=np.int32)
        sims = np.empty(cap, dtype=np.float64)
        n = C.c_int32(0)
        _check(knn_lib().rs_knn_predict_neighbors(self.h, int(left), int(right), cap, _ptr(ids), _ptr(sims),
                                                  C.byref(n)))
        return ids[:n.value].copy(), sims[:n.value].copy()

    def sims_rows(self, row0, nrows):
        out = np.empty((nrows, self.n_left), dtype=np.float64)
        _check(knn_lib().rs_knn_sims_rows(self.h, row0, nrows, _ptr(out)))
        return out

    def topk(self, k):
        rows = self.rows[1] - self.rows[0]
        idx = np.empty((rows, k), dtype=np.int32)
        sim = np.empty((rows, k), dtype=np.float64)
        _check(knn_lib().rs_knn_topk(self.h, k, _ptr(idx), _ptr(sim)))
        return idx, sim

    def topk_device(self, k, d_idx, d_sim):
        _check(knn_lib().rs_knn_topk_device(self.h, k, d_idx, d_sim))

    def cosums(self, row0, nrows):
        out = np.empty((nrows, self.n_left, 6), dtype=np.int32)
        _check(knn_lib().rs_knn_cosums(self.h, row0, nrows, _ptr(out)))
        return out

    def means(self):
        out = np.empty(self.n_left, dtype=np.float64)
        _check(knn_lib().rs_knn_means(self.h, _ptr(out)))
        return out

    def stddevs(self):
        out = np.empty(self.n_left, dtype=np.float64)
        _check(knn_lib().rs_knn_stddevs(self.h, _ptr(out)))
        return out

    def profile(self):
        p = RsKnnProfile()
        _check(knn_lib().rs_knn_profile_get(self.h, C.byref(p)))
        return {f: getattr(p, f) for f, _ in RsKnnProfile._fields_ if f != "reserved0"}

    def profile_reset(self):
        _check(knn_lib().rs_knn_profile_reset(self.h))

    def synchronize(self):
        _check(knn_lib().rs_knn_synchronize(self.h))

    def set_k(self, k, min_k):
        _check(knn_lib().rs_knn_set_k(self.h, int(k), int(min_k)))

    def _n_targets(self, side):
        return self.n_left if side == RS_SIDE["right"] else self.n_right

    def score_all(self, side, queries):
        """Full score rows [len(queries)][n_targets] of inner-id queries of `side` ("left" / "right"); rated
        targets NaN (include/rs_knn.h rs_knn_score_all)."""
        side = RS_SIDE[side]
        q = np.ascontiguousarray(queries, dtype=np.int32)
        out = np.empty((len(q), self._n_targets(side)), dtype=np.float64)
        _check(knn_lib().rs_knn_score_all(self.h, side, _ptr(q), len(q), _ptr(out)))
        return out

    def score_all_device(self, side, d_queries, n, d_out):
        _check(knn_lib().rs_knn_score_all_device(self.h, RS_SIDE[side], d_queries, n, d_out))

    def recommend(self, side, queries, n_top):
        """(ids[len(queries)][n_top], scores[len(queries)][n_top]): the n_top best unrated targets of each
        inner-id query (include/rs_knn.h rs_knn_recommend)."""
        side = RS_SIDE[side]
        q = np.ascontiguousarray(queries, dtype=np.int32)
        ids = np.empty((len(q), n_top), dtype=np.int32)
        scores = np.empty((len(q), n_top), dtype=np.float64)
        _check(knn_lib().rs_knn_recommend(self.h, side, _ptr(q), len(q), int(n_top), _ptr(ids), _ptr(scores)))
        return ids, scores

    def recommend_device(self, side, d_queries, n, n_top, d_ids, d_scores):
        _check(knn_lib().rs_knn_recommend_device(self.h, RS_SIDE[side], d_queries, n, int(n_top), d_ids, d_scores))

    def score_all_sharded_device(self, side, d_queries, n, d_out):
        """Row shards: the score rows of this shard, +0.0 in the cells it does not answer (include/rs_knn.h
        rs_knn_score_all_sharded_device); an integer sum of the shards' bit patterns is rs_knn_score_all."""
        _check(knn_lib().rs_knn_score_all_sharded_device(self.h, RS_SIDE[side], d_queries, n, d_out))

    def recommend_sharded_device(self, side, d_queries, n, n_top, d_ids, d_scores):
        """Row shards: the partial top-n_top lists of this shard, to be united across the shards
        (shard.union_recommend_device)."""
        _check(knn_lib().rs_knn_recommend_sharded_device(self.h, RS_SIDE[side], d_queries, n, int(n_top), d_ids,
                                                         d_scores))

    @staticmethod
    def _given_lists(ptr, ids, vals):
        ptr = np.ascontiguousarray(ptr, dtype=np.int64)
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        if len(ids) == 0:           # the library wants valid pointers even when every list is empty
            ids, vals = np.zeros(1, np.int32), np.zeros(1, np.float64)
        return ptr, ids, vals, len(ptr) - 1

    def score_all_given(self, side, ptr, ids, vals):
        """Full score rows [n][n_targets] of queries given as rating lists: list b is ids[ptr[b]:ptr[b+1]] (inner ids
        of the target side) with ratings vals[...] (include/rs_knn.h rs_knn_score_all_given)."""
        side = RS_SIDE[side]
        ptr, ids, vals, n = self._given_lists(ptr, ids, vals)
        out = np.empty((n, self._n_targets(side)), dtype=np.float64)
        _check(knn_lib().rs_knn_score_all_given(self.h, side, _ptr(ptr), _ptr(ids), _ptr(vals), n, _ptr(out)))
        return out

    def score_all_given_device(self, side, d_ptr, d_ids, d_vals, n, d_out):
        _check(knn_lib().rs_knn_score_all_given_device(self.h, RS_SIDE[side], d_ptr, d_ids, d_vals, n, d_out))

    def recommend_given(self, side, ptr, ids, vals, n_top):
        """(ids[n][n_top], scores[n][n_top]) of queries given as rating lists (rs_knn_recommend_given)."""
        side = RS_SIDE[side]
        ptr, ids, vals, n = self._given_lists(ptr, ids, vals)
        top_ids = np.empty((n, n_top), dtype=np.int32)
        top = np.empty((n, n_top), dtype=np.float64)
        _check(knn_lib().rs_knn_recommend_given(self.h, side, _ptr(ptr), _ptr(ids), _ptr(vals), n, int(n_top),
                                                _ptr(top_ids), _ptr(top)))
        return top_ids, top

    def recommend_given_device(self, side, d_ptr, d_ids, d_vals, n, n_top, d_top_ids, d_top_scores):
        _check(knn_lib().rs_knn_recommend_given_device(self.h, RS_SIDE[side], d_ptr, d_ids, d_vals, n, int(n_top),
                                                       d_top_ids, d_top_scores))

    # ---- cyclic row shards (RS_STORE_MATRIX, shard_count >= 2): the exchange step ----
    def peer_export(self):
        """(64-byte CUDA IPC handle, byte offset) of this shard's matrix."""
        hb = np.zeros(64, dtype=np.uint8)
        off = C.c_int64(0)
        _check(knn_lib().rs_knn_peer_export(self.h, _ptr(hb), C.byref(off)))
        return hb, int(off.value)

    def peer_import(self, handles, offsets):
        handles = np.ascontiguousarray(handles, dtype=np.uint8).reshape(-1, 64)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        _check(knn_lib().rs_knn_peer_import(self.h, len(offsets), _ptr(handles), _ptr(offsets)))

    def peer_import_local(self, peers):
        arr = (C.c_void_p * len(peers))(*[p.h for p in peers])
        _check(knn_lib().rs_knn_peer_import_local(self.h, len(peers), arr))

    def mirror(self):
        _check(knn_lib().rs_knn_mirror(self.h))

    def owned_rows(self):
        """Global ids of the left rows this handle stores, in storage order."""
        if self.params.store == RS_STORE["matrix"] and self.params.shard_count >= 2:
            return cyclic_rows(self.n_left, self.params.shard_count, self.params.shard_index)
        return np.arange(self.rows[0], self.rows[1])


# --------------------------------------------------------------------------------------------
# core/base.go:108-163 — BaseLine (host; sequential SGD)
# --------------------------------------------------------------------------------------------
class Base:
    """core/base.go:59-74"""

    def __init__(self, params=None):
        self.Params = _params(params)
        self.Data = None

    def SetParams(self, params):
        self.Params = _params(params)

    def Predict(self, userId, itemId):
        raise NotImplementedError("Predict() not implemented")  # core/base.go:68-70 panics

    def Fit(self, trainSet):
        raise NotImplementedError("Fit() not implemented")


class BaseLine(Base):
    def Fit(self, trainSet: TrainSet):
        reg = self.Params.GetFloat64("reg", 0.02)
        lr = self.Params.GetFloat64("lr", 0.005)
        nEpochs = self.Params.GetInt("nEpochs", 20)
        self.trainSet = trainSet
        self.userBias = np.zeros(trainSet.UserCount, dtype=np.float64)
        self.itemBias = np.zeros(trainSet.ItemCount, dtype=np.float64)
        if self.Params.GetString("baseline", "sgd") == "als":
            # EXTENSION (BASELINE.json config 3): ALS baselines on the device, rs_baseline_als
            iu = np.ascontiguousarray(trainSet.innerUsers, dtype=np.int32)
            ii = np.ascontiguousarray(trainSet.innerItems, dtype=np.int32)
            rr = np.ascontiguousarray(trainSet.Ratings, dtype=np.float64)
            _check(knn_lib().rs_baseline_als(self.Params.GetInt("device", -1), _ptr(iu), _ptr(ii), _ptr(rr),
                                             len(rr), trainSet.UserCount, trainSet.ItemCount,
                                             trainSet.GlobalMean, self.Params.GetFloat64("regU", 15.0),
                                             self.Params.GetFloat64("regI", 10.0),
                                             self.Params.GetInt("nEpochs", 10), _ptr(self.userBias),
                                             _ptr(self.itemBias)))
            self.globalBias = trainSet.GlobalMean
            return
        gb = C.c_double(0.0)
        host_lib().rs_host_baseline_sgd(_ptr(trainSet.innerUsers), _ptr(trainSet.innerItems),
                                        _ptr(trainSet.Ratings), trainSet.Length(), trainSet.UserCount,
                                        trainSet.ItemCount, reg, lr, nEpochs, _ptr(self.userBias),
                                        _ptr(self.itemBias), C.byref(gb))
        self.globalBias = gb.value

    def Predict(self, userId, itemId):
        """core/base.go:122-134"""
        iu = self.trainSet.ConvertUserID(userId)
        ii = self.trainSet.ConvertItemID(itemId)
        ret = self.globalBias
        if iu != newID:
            ret += self.userBias[iu]
        if ii != newID:
            ret += self.itemBias[ii]
        return ret


def NewBaseLine(params=None):
    return BaseLine(params)


# --------------------------------------------------------------------------------------------
# core/knn.go — KNN
# --------------------------------------------------------------------------------------------
class KNN(Base):
    """core/knn.go:17-27.  `Sims`, `Means`, `StdDevs`, `Bias` stay available as in the reference
    (Sims is materialised from the device on demand)."""

    # extra Parameters keys understood by the device path (SURVEY.md §5 "Config / flags")
    _DEVICE_KEYS = ("device", "pearsonMode", "simPath", "store", "topk", "rowBegin", "rowEnd", "shrinkage",
                    "baseline", "regU", "regI", "shardCount", "shardIndex")

    def __init__(self, knn_type, params=None):
        super().__init__(params)
        self.KNNType = knn_type  # core/knn.go:50-73: fixed by the constructor
        self.GlobalMean = math.nan
        self.Means = None
        self.StdDevs = None
        self.Bias = None
        self._h = None

    def Close(self):
        if self._h is not None:
            self._h.close()
            self._h = None

    def __del__(self):
        self.Close()

    def _prepare(self, trainSet: TrainSet):
        """The host half of core/knn.go:143-187: parameters, orientation, baseline biases."""
        sim = self.Params.GetSim("sim", MSD)
        userBased = self.Params.GetBool("userBased", True)
        self.Params.GetInt("nJobs", 0)  # accepted for compatibility; the device needs no job count
        self.Data = trainSet
        self.GlobalMean = trainSet.GlobalMean
        if userBased:
            left, right, n_left, n_right = trainSet.innerUsers, trainSet.innerItems, trainSet.UserCount, trainSet.ItemCount
        else:
            left, right, n_left, n_right = trainSet.innerItems, trainSet.innerUsers, trainSet.ItemCount, trainSet.UserCount
        left_bias = right_bias = None
        global_bias = 0.0
        if self.KNNType == baseline or sim.name == "pearson_baseline":
            bl = NewBaseLine(self.Params)           # core/knn.go:179-187
            bl.Fit(trainSet)
            ub, ib = bl.userBias, bl.itemBias
            left_bias, right_bias = (ub, ib) if userBased else (ib, ub)
            global_bias = bl.globalBias
            if self.KNNType == baseline:
                self.Bias = left_bias
            if sim.name != "pearson_baseline":
                right_bias = None
        self._userBased = userBased
        return sim, left, right, n_left, n_right, left_bias, right_bias, global_bias

    def _new_handle(self, sim, **over):
        k = self.Params.GetInt("k", 40)
        minK = self.Params.GetInt("mink", 1)
        self._kk = (k, minK)
        kw = dict(sim=sim.name, knn_type=self.KNNType, k=k, min_k=minK,
                  device=self.Params.GetInt("device", -1),
                  pearson_mode=self.Params.GetString("pearsonMode", "exact"),
                  sim_path=self.Params.GetString("simPath", "auto"),
                  store=self.Params.GetString("store", "matrix"),
                  topk=self.Params.GetInt("topk", 0),
                  row_begin=self.Params.GetInt("rowBegin", 0), row_end=self.Params.GetInt("rowEnd", 0),
                  shrinkage=self.Params.GetFloat64("shrinkage", 0.0),
                  shard_count=self.Params.GetInt("shardCount", 0),
                  shard_index=self.Params.GetInt("shardIndex", 0))
        kw.update(over)
        return _Handle(**kw)

    def _after_fit(self):
        if self.KNNType in (centered, zScore):
            self.Means = self._h.means()
        if self.KNNType == zScore:
            self.StdDevs = self._h.stddevs()

    def Fit(self, trainSet: TrainSet):
        """core/knn.go:143-217"""
        sim, left, right, n_left, n_right, left_bias, right_bias, global_bias = self._prepare(trainSet)
        self.Close()
        self._h = self._new_handle(sim)
        self._h.fit(left, right, trainSet.Ratings, n_left, n_right, trainSet.GlobalMean, left_bias, right_bias,
                    global_bias)
        self._after_fit()

    def Update(self, rowSet: DataSet):
        """Adds the ratings of `rowSet` (raw user, raw item, rating; users and items may be new) to the fitted model
        without a refit: the model becomes the Fit of Data.Extend(rowSet), bit for bit — similarities, Means, StdDevs,
        GlobalMean, Predict and Recommend (rs_knn_update; only the rows of the users (items) the ratings touch are
        recomputed).  A pair the model already holds is refused, as are models an update cannot extend exactly:
        KNNBaseline, PearsonBaseline, Pearson in sums mode, row shards, top-k-only stores."""
        data = self.Data.Extend(rowSet)
        n0 = self.Data.Length()
        iu, ii = data.innerUsers[n0:], data.innerItems[n0:]
        if self._userBased:
            left, right, n_left, n_right = iu, ii, data.UserCount, data.ItemCount
        else:
            left, right, n_left, n_right = ii, iu, data.ItemCount, data.UserCount
        self._h.update(left, right, data.Ratings[n0:], n_left, n_right, data.GlobalMean)
        self.Data = data
        self.GlobalMean = data.GlobalMean
        self._after_fit()

    @property
    def Sims(self):
        """core/knn.go:21 — the dense N x N matrix, NaN = unset (copied from HBM on demand)."""
        if self._h.params.store == RS_STORE["matrix"] and self._h.params.shard_count >= 2:
            rows = self._h.owned_rows()          # cyclic shard: block by block, in storage order
            return np.concatenate([self._h.sims_rows(int(b[0]), len(b))
                                   for b in np.split(rows, np.flatnonzero(np.diff(rows) != 1) + 1)])
        r0, r1 = self._h.rows
        return self._h.sims_rows(r0, r1 - r0)

    def PredictBatch(self, userIDs, itemIDs):
        """BatchPredictor: the whole of DataSet.Predict (core/data.go:98-105) in one device call."""
        # large batches: the inner ids are written into page-locked staging memory (and the predictions come back
        # into it): both copies of rs_knn_predict_batch then run at full PCIe speed
        big = len(userIDs) >= 1 << 16
        iu = self.Data.convert_users(userIDs, out=pinned_empty(len(userIDs), np.int32) if big else None)
        ii = self.Data.convert_items(itemIDs, out=pinned_empty(len(itemIDs), np.int32) if big else None)
        left, right = (iu, ii) if self._userBased else (ii, iu)
        self._sync_k()
        return self._h.predict_batch(left, right)

    def Predict(self, userID, itemID):
        """core/knn.go:75-141 (a one-element batch)."""
        return float(self.PredictBatch(np.array([userID]), np.array([itemID]))[0])

    def Neighbors(self, userID, itemID):
        """The neighbours Predict used for this pair, in accumulation order (inner ids, sims)."""
        iu = self.Data.ConvertUserID(userID)
        ii = self.Data.ConvertItemID(itemID)
        if iu == newID or ii == newID:
            return np.empty(0, np.int32), np.empty(0, np.float64)
        left, right = (iu, ii) if self._userBased else (ii, iu)
        return self._h.predict_neighbors(left, right)

    def TopK(self, k):
        return self._h.topk(k)

    def _sync_k(self):
        # core/knn.go:80-81 reads k / mink in Predict: SetParams after Fit takes effect here
        k, mink = self.Params.GetInt("k", 40), self.Params.GetInt("mink", 1)
        if (k, mink) != self._kk:
            self._h.set_k(k, mink)
            self._kk = (k, mink)

    def _user_queries(self, userIDs):
        self._sync_k()
        side = "left" if self._userBased else "right"
        return side, self.Data.convert_users(np.asarray(userIDs, dtype=np.int64))

    def ScoreAll(self, userIDs):
        """The score of every item for each user, [len(userIDs)][ItemCount] in inner item order: Predict(user, item)
        bit for bit, NaN for the items the user rated (an unknown user scores GlobalMean everywhere)."""
        side, q = self._user_queries(userIDs)
        return self._h.score_all(side, q)

    def Recommend(self, userIDs, n):
        """(items[len][n], scores[len][n]): the n best items each user has not rated, by (score desc, inner item id
        asc), as raw item ids; unused slots are newID (-1) with score NaN."""
        side, q = self._user_queries(userIDs)
        ids, scores = self._h.recommend(side, q, n)
        return self._raw_items(ids), scores

    def _given(self, dataSet):
        """(users, ptr, ids, vals): the rows of `dataSet` grouped by raw user in order of first appearance, each
        user's entries in dataset order, as lists of inner item ids.  Items the train set does not know are dropped:
        they have no row or column of the model, so Predict could never use them (nor do they enter the list's mean
        on the user-based side).  A user all of whose items are unknown keeps an empty list (GlobalMean)."""
        users = np.asarray(dataSet.Users, dtype=np.int64)
        uniq, first, inv = np.unique(users, return_index=True, return_inverse=True)
        rank = np.empty(len(uniq), dtype=np.int64)
        rank[np.argsort(first, kind="stable")] = np.arange(len(uniq))
        grp = rank[inv.reshape(-1)]
        inner = self.Data.convert_items(np.asarray(dataSet.Items, dtype=np.int64))
        keep = inner >= 0
        order = np.argsort(grp[keep], kind="stable")
        ids = inner[keep][order]
        vals = np.asarray(dataSet.Ratings, dtype=np.float64)[keep][order]
        ptr = np.zeros(len(uniq) + 1, dtype=np.int64)
        np.cumsum(np.bincount(grp[keep], minlength=len(uniq)), out=ptr[1:])
        return uniq[np.argsort(first, kind="stable")], ptr, ids, vals

    def ScoreAllGiven(self, dataSet):
        """Fold-in: (users, scores[len(users)][ItemCount]) for users whose ratings are given in `dataSet` (raw user,
        raw item, rating) instead of taken from the train set — users who may or may not be in it.  The scores are
        those of ScoreAll for a user whose ratings are the given ones; the model is not refitted (the given ratings
        enter neither the similarities between the train set's rows, nor its means, nor GlobalMean)."""
        self._sync_k()
        users, ptr, ids, vals = self._given(dataSet)
        return users, self._h.score_all_given("left" if self._userBased else "right", ptr, ids, vals)

    def RecommendGiven(self, dataSet, n):
        """Fold-in: (users, items[len][n], scores[len][n]) — Recommend for users whose ratings are given in `dataSet`
        (see ScoreAllGiven); the given items are never recommended."""
        self._sync_k()
        users, ptr, ids, vals = self._given(dataSet)
        top_ids, top = self._h.recommend_given("left" if self._userBased else "right", ptr, ids, vals, n)
        return users, self._raw_items(top_ids), top

    def _raw_items(self, ids):
        """Inner item ids -> raw item ids; -1 (an unused slot) -> newID."""
        raw = np.empty(self.Data.ItemCount, dtype=np.int64)    # inner -> raw: the order of first appearance
        raw[self.Data.innerItems] = self.Data.Items
        return np.where(ids >= 0, raw[np.maximum(ids, 0)], newID)

    def Profile(self):
        return self._h.profile()


def NewKNN(params=None):
    return KNN(basic, params)


def NewKNNWithMean(params=None):
    return KNN(centered, params)


def NewKNNWithZScore(params=None):
    return KNN(zScore, params)


def NewKNNBaseLine(params=None):
    return KNN(baseline, params)


# --------------------------------------------------------------------------------------------
# core/slope_one.go — Slope One (SURVEY.md §8 f-2: the step next to the KNN path)
# --------------------------------------------------------------------------------------------
class SlopeOne(Base):
    """core/slope_one.go:8-14.  Fit builds the item x item deviation matrix on the device (the same
    co-rated integer contractions as the KNN similarities: count, sum r_i, sum r_j on the tensor
    cores); Predict is a gather over the user's ratings.  `dev` and `userMeans` stay available."""

    def __init__(self, params=None):
        super().__init__(params)
        self.globalMean = math.nan
        self.userMeans = None
        self._h = None

    def Close(self):
        if self._h is not None:
            self._h.close()
            self._h = None

    def __del__(self):
        self.Close()

    def Fit(self, trainSet: TrainSet):
        """core/slope_one.go:47-93"""
        self.Data = trainSet
        self.globalMean = trainSet.GlobalMean
        self.Close()
        self._h = _Handle(sim="slope_one", knn_type="basic", device=self.Params.GetInt("device", -1),
                          row_begin=self.Params.GetInt("rowBegin", 0), row_end=self.Params.GetInt("rowEnd", 0))
        self._h.fit(trainSet.innerItems, trainSet.innerUsers, trainSet.Ratings, trainSet.ItemCount,
                    trainSet.UserCount, trainSet.GlobalMean)

    @property
    def dev(self):
        """core/slope_one.go:13 — the item x item deviation matrix (copied from HBM on demand)."""
        if self._h.params.store == RS_STORE["matrix"] and self._h.params.shard_count >= 2:
            rows = self._h.owned_rows()          # cyclic shard: block by block, in storage order
            return np.concatenate([self._h.sims_rows(int(b[0]), len(b))
                                   for b in np.split(rows, np.flatnonzero(np.diff(rows) != 1) + 1)])
        r0, r1 = self._h.rows
        return self._h.sims_rows(r0, r1 - r0)

    def PredictBatch(self, userIDs, itemIDs):
        iu = self.Data.convert_users(userIDs)
        ii = self.Data.convert_items(itemIDs)
        return self._h.predict_batch(ii, iu)

    def Predict(self, userID, itemID):
        """core/slope_one.go:22-45 (a one-element batch)."""
        return float(self.PredictBatch(np.array([userID], dtype=np.int64), np.array([itemID], dtype=np.int64))[0])


def NewSlopeOne(params=None):
    """core/slope_one.go:16-20 (the reference drops `params`; nothing in Slope One reads any)."""
    return SlopeOne(params)


# --------------------------------------------------------------------------------------------
# core/utils.go:160-180 + core/eval.go:18-67 — metrics and CrossValidate (intended signatures)
# --------------------------------------------------------------------------------------------
def RMSE(predictions, truth):
    predictions = np.asarray(predictions, dtype=np.float64)
    truth = np.asarray(truth, dtype=np.float64)
    return float(np.sqrt(np.sum((predictions - truth) * (predictions - truth)) / len(truth)))


def MAE(predictions, truth):
    predictions = np.asarray(predictions, dtype=np.float64)
    truth = np.asarray(truth, dtype=np.float64)
    return float(np.sum(np.abs(predictions - truth)) / len(truth))


class CrossValidateResult:
    def __init__(self, cv):
        self.Trains = [0.0] * cv
        self.Tests = [0.0] * cv


def CrossValidate(estimator, dataSet, metrics, cv, seed, params):
    """core/eval.go:18-67 with the 6-argument form every caller uses (SURVEY.md §4.3).  Each fold
    works on its own copy of the estimator (the reference gob-copies it, core/eval.go:29-30) and
    REPLACES its Params with `params` (core/eval.go:34)."""
    ret = [CrossValidateResult(cv) for _ in metrics]
    trainFolds, testFolds = dataSet.KFold(cv, seed)
    for i in range(cv):
        cp = type(estimator).__new__(type(estimator))
        cp.__dict__.update({k: v for k, v in estimator.__dict__.items() if k != "_h"})
        cp._h = None
        cp.SetParams(params)
        cp.Fit(trainFolds[i])
        testPredictions = testFolds[i].Predict(cp)
        for j, metric in enumerate(metrics):
            ret[j].Tests[i] = metric(testPredictions, testFolds[i].Ratings)
        if hasattr(cp, "Close"):
            cp.Close()
    return ret


def synth_ratings(n_users, n_items, nnz, seed):
    """Deterministic synthetic COO of a BASELINE.json shape (host/rs_host.cc)."""
    users = np.empty(nnz, dtype=np.int64)
    items = np.empty(nnz, dtype=np.int64)
    ratings = np.empty(nnz, dtype=np.float64)
    w = host_lib().rs_host_synth_ratings(n_users, n_items, nnz, seed, _ptr(users), _ptr(items), _ptr(ratings))
    return DataSet(users[:w], items[:w], ratings[:w])
