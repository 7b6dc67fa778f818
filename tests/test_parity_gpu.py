"""Parity of the CUDA path against the oracle, through the C ABI (run with -m gpu on a B200).

Bar (BASELINE.json north_star): neighbour indices bit-exact (ties broken by inner id),
similarities and predictions within 1e-9 relative for float64 — here they are in fact required
to be BIT-IDENTICAL wherever the device path replays the reference's operation order (every
path except Pearson in `sums` mode, which is held to 1e-9*max(1,|ref|))."""
import numpy as np
import pytest

import recommend_sys_b200 as rs
from oracle import binding as ob
from conftest import bits_equal, split

pytestmark = pytest.mark.gpu

A = rs.NewSortedIdRatings([(1, 4), (2, 5), (3, 6)])   # core/sim_test.go:11-20
B = rs.NewSortedIdRatings([(0, 0), (1, 1), (2, 2)])


# ---- the reference's own known-answer tests, replayed on the device ----
@pytest.mark.parametrize("path", ["stream", "auto"])
def test_cosine(path):   # core/sim_test.go:10-25
    assert rs.Cosine(A, B, sim_path=path) == 0.9778024140774094


@pytest.mark.parametrize("path", ["stream", "auto"])
def test_msd(path):      # core/sim_test.go:27-42
    assert rs.MSD(A, B, sim_path=path) == 0.1


def test_pearson():      # core/sim_test.go:44-59
    assert rs.Pearson(A, B) == 0.0


def test_no_corating_is_nan():
    a, b = rs.NewSortedIdRatings([(1, 4)]), rs.NewSortedIdRatings([(2, 3)])
    for sim in (rs.Cosine, rs.MSD, rs.Pearson):
        assert np.isnan(sim(a, b))


SIMS = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson}
CTORS = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore,
         "baseline": rs.NewKNNBaseLine}


def fit_pair(train_arr, sim, knn_type, user_based, k=40, mink=1, extra=None):
    u, i, r = split(train_arr)
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    params = {"sim": SIMS[sim], "userBased": user_based, "k": k, "mink": mink}
    params.update(extra or {})
    est = CTORS[knn_type](rs.Parameters(params))
    est.Fit(ts)
    ots = ob.TrainSet(u, i, r)
    ref = ob.KNN(sim=sim, knn_type=knn_type, user_based=user_based, k=k, min_k=mink, n_jobs=8,
                 tie_policy="canonical").fit(ots)
    return est, ref


# ---- similarity matrix: every sim x both orientations on the real ml-100k fold u1 ----
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd", "pearson"])
def test_sims_bit_exact_ml100k(ml100k, sim, user_based):
    est, ref = fit_pair(ml100k["u1_base"], sim, "basic", user_based, extra={"simPath": "stream"})
    got, want = est.Sims, ref.sims()
    assert got.shape == want.shape
    assert np.isnan(np.diag(got)).all()                      # core/knn.go:202
    assert bits_equal(got, want)
    assert bits_equal(got, got.T)                            # core/knn.go:205-208


# ---- both triangles of the full-matrix stream Fit (rs_prep_rt picks the cheaper one per Fit) ----
@pytest.mark.parametrize("tri", ["upper", "lower"])
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd", "pearson"])
def test_sims_bit_exact_both_triangles(ml100k, sim, user_based, tri, monkeypatch):
    monkeypatch.setenv("RS_KNN_STREAM_TRI", tri)
    est, ref = fit_pair(ml100k["u4_base"], sim, "basic", user_based, extra={"simPath": "stream"})
    got, want = est.Sims, ref.sims()
    assert np.isnan(np.diag(got)).all()
    assert bits_equal(got, want)
    assert bits_equal(got, got.T)


# ---- cyclic row shards (the multi-GPU Fit + Predict): every shard computes one triangle of its rows,
# the mirror step pulls the other one from the peers; here all shards live on one GPU ----
# pop_min "200": the longer rows are popular columns (mirror_pop_kernel); None: ML-100K has no row of the default
# 8192 entries, so there are none and the plain column walk is mirrored by mirror_kernel
@pytest.mark.parametrize("pop_min", ["200", None])
@pytest.mark.parametrize("tri", ["upper", "lower"])
@pytest.mark.parametrize("count", [2, 3])
def test_cyclic_row_shards_equal_full(ml100k, count, tri, pop_min, monkeypatch):
    monkeypatch.setenv("RS_KNN_STREAM_TRI", tri)
    monkeypatch.setenv("RS_KNN_STREAM_JC", "256")
    if pop_min is None:
        monkeypatch.delenv("RS_KNN_POP_MIN", raising=False)
    else:
        monkeypatch.setenv("RS_KNN_POP_MIN", pop_min)
    u, i, r = split(ml100k["u1_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    base = {"sim": rs.Pearson, "userBased": False, "k": 40}
    full = rs.NewKNNWithMean(rs.Parameters(base))
    full.Fit(ts)
    want = full.Sims
    ref = ob.KNN(sim="pearson", knn_type="centered", user_based=False, k=40, n_jobs=8,
                 tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    assert bits_equal(want, ref.sims())
    tu, ti, _ = split(ml100k["u1_test"])
    want_pred = full.PredictBatch(tu, ti)
    shards = []
    for q in range(count):
        est = rs.NewKNNWithMean(rs.Parameters(dict(base, shardCount=count, shardIndex=q)))
        est.Fit(ts)
        shards.append(est)
    with pytest.raises(rs.core.RsError):          # one triangle only until the mirror step has run
        shards[0].PredictBatch(tu[:4], ti[:4])
    for est in shards:
        est._h.synchronize()
    for est in shards:
        est._h.peer_import_local([x._h for x in shards])
        est._h.mirror()
    got_pred = np.full(len(tu), np.nan)
    left = ts.convert_items(ti)
    owner = rs.shard.route_pairs(left, count)
    for q, est in enumerate(shards):
        rows = est._h.owned_rows()
        assert bits_equal(est.Sims, want[rows]), (q, count, tri)
        mine = np.flatnonzero(owner == q)
        got_pred[mine] = est.PredictBatch(tu[mine], ti[mine])
        other = np.flatnonzero((owner != q) & (left >= 0))[:16]
        assert np.isnan(est.PredictBatch(tu[other], ti[other])).all()     # rows of another shard: NaN
    assert bits_equal(got_pred, want_pred)
    assert sorted(np.concatenate([e._h.owned_rows() for e in shards]).tolist()) == list(range(want.shape[0]))
    # the all-reduce form: every shard gets the FULL test set (plus cold-start pairs), answers its own pairs and
    # leaves +0.0 elsewhere; the integer sum of the bit patterns over the shards is the complete vector
    import torch

    tu2 = np.concatenate([tu, [10 ** 9, 10 ** 9 + 1, 10 ** 9 + 2]])       # unknown users and items
    ti2 = np.concatenate([ti, [int(ti[0]), 10 ** 9, int(ti[1])]])
    want2 = full.PredictBatch(tu2, ti2)
    d_l = torch.from_numpy(ts.convert_items(ti2).astype(np.int32)).cuda()
    d_r = torch.from_numpy(ts.convert_users(tu2).astype(np.int32)).cuda()
    acc = np.zeros(len(tu2), dtype=np.int64)
    for est in shards:
        d_o = torch.empty(len(tu2), dtype=torch.float64, device="cuda")
        est._h.predict_batch_sharded_device(d_l.data_ptr(), d_r.data_ptr(), len(tu2), d_o.data_ptr())
        est._h.synchronize()
        acc += d_o.cpu().numpy().view(np.int64)
    assert bits_equal(acc.view(np.float64), want2)
    for est in shards:
        est.Close()


def test_save_load_estimator_and_neighbor_lists(ml100k, tmp_path):
    # core/dump_test.go:9-29 (TestSave) for the estimators of this path: the restored model predicts the same
    u, i, r = split(ml100k["u4_base"])
    tu, ti, tr = split(ml100k["u4_test"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    est1 = rs.NewKNNWithZScore(rs.Parameters({"sim": rs.Pearson, "userBased": False, "k": 30}))
    est1.Fit(ts)
    err1 = rs.RMSE(np.nan_to_num(rs.NewRawSet(tu, ti, tr).Predict(est1)), tr)
    rs.Save(tmp_path / "m" / "knn.m", est1)
    est2 = rs.Load(tmp_path / "m" / "knn.m")
    p1, p2 = rs.NewRawSet(tu, ti, tr).Predict(est1), rs.NewRawSet(tu, ti, tr).Predict(est2)
    assert bits_equal(p1, p2) and err1 == rs.RMSE(np.nan_to_num(p2), tr)
    assert est2.KNNType == "zscore" and est2.Params["sim"] is rs.Pearson and bits_equal(est1.StdDevs, est2.StdDevs)
    # the neighbour lists of a top-k-only Fit, device -> file -> host
    idx, sim = est1.TopK(25)
    rs.SaveNeighbors(tmp_path / "lists.rsknn", idx, sim)
    i2, s2 = rs.LoadNeighbors(tmp_path / "lists.rsknn")
    assert np.array_equal(idx, i2) and bits_equal(sim, s2)
    so = rs.NewSlopeOne(None)
    so.Fit(ts)
    rs.Save(tmp_path / "so.m", so)
    assert bits_equal(rs.NewRawSet(tu, ti, tr).Predict(so), rs.NewRawSet(tu, ti, tr).Predict(rs.Load(tmp_path / "so.m")))


def test_cpp_host_mirror_benchmark_on_ml100k(ml100k, tmp_path):
    """host/core.hpp + host/benchmark.cc — the compiled mirror of the reference's Go API and of benchmark.go —
    run end to end over the same C ABI on the real MovieLens-100K: 5-fold cross-validation with params = nil,
    held to the reference's own acceptance bounds (core/base_test.go:46-64, RMSE/MAE <= expect + 0.008)."""
    import subprocess
    from pathlib import Path

    exe = Path(rs.core.__file__).resolve().parent / "rs_benchmark"
    assert exe.exists(), "run __graft_entry__.build() (host/Makefile builds rs_benchmark)"
    data = tmp_path / "u.data"
    np.savetxt(data, ml100k["u_data"][:, :3], fmt="%d", delimiter="\t")
    out = subprocess.run([str(exe), str(data)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    rows = {}
    for line in out.stdout.splitlines()[1:]:
        parts = line.rsplit(None, 3)
        rows[parts[0].strip()] = (float(parts[1]), float(parts[2]))
    bounds = {"KNN": (0.980, 0.774), "Centered K-NN": (0.951, 0.749), "K-NN Z-Score": (0.951, 0.746),
              "K-NN Baseline": (0.931, 0.733), "Slope One": (0.946, 0.743)}
    for name, (rmse, mae) in bounds.items():
        assert rows[name][0] <= rmse + 0.008 and rows[name][1] <= mae + 0.008, (name, rows[name])


def test_k_is_read_at_predict_time(ml100k):
    # core/knn.go:80-81: k / mink are read by Predict, so SetParams after Fit changes the answer
    est, ref = fit_pair(ml100k["u2_base"], "msd", "basic", True, k=40)
    _, ref10 = None, None
    u, i, r = split(ml100k["u2_test"])
    before = est.PredictBatch(u, i)
    est.Params["k"] = 10
    after = est.PredictBatch(u, i)
    est10, ref10 = fit_pair(ml100k["u2_base"], "msd", "basic", True, k=10)
    assert bits_equal(after, ref10.predict_batch(u, i, n_threads=8))
    assert not bits_equal(before, after)


def test_concurrent_predict_on_one_handle(ml100k):
    # the reference's Predict is read-only and goroutine-safe; calls on one handle are serialised here
    import threading

    est, ref = fit_pair(ml100k["u3_base"], "cosine", "basic", True)
    u, i, r = split(ml100k["u3_test"])
    want = ref.predict_batch(u, i, n_threads=8)
    parts = np.array_split(np.arange(len(u)), 8)
    out = [None] * len(parts)

    def work(t):
        for _ in range(5):
            out[t] = est.PredictBatch(u[parts[t]], i[parts[t]])

    ths = [threading.Thread(target=work, args=(t,)) for t in range(len(parts))]
    [t.start() for t in ths]
    [t.join() for t in ths]
    assert bits_equal(np.concatenate(out), want)


# ---- page-locked staging of large batches (rs_knn_host_alloc): same predictions as the pageable path, blocks are
# cached and reused ----
def test_pinned_staging_of_large_batches(ml100k):
    import ctypes as C

    L = rs.core.knn_lib()
    p, q = C.c_void_p(), C.c_void_p()
    assert L.rs_knn_host_alloc(1 << 20, C.byref(p)) == 0 and p.value
    assert L.rs_knn_host_free(p) == 0
    assert L.rs_knn_host_alloc(1 << 20, C.byref(q)) == 0 and q.value == p.value      # reused
    assert L.rs_knn_host_free(q) == 0
    assert L.rs_knn_host_free(C.c_void_p(12345)) != 0
    arr = rs.core.pinned_empty(1000, np.float64)
    arr[:] = np.arange(1000)
    assert arr.base is not None and arr.sum() == 499500.0
    u, i, r = split(ml100k["u1_base"])
    est = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False, "k": 40}))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    tu, ti, _ = split(ml100k["u1_test"])
    small = np.concatenate([est.PredictBatch(tu[x:x + 5000], ti[x:x + 5000]) for x in range(0, len(tu), 5000)])
    big_u, big_i = np.tile(tu, 4), np.tile(ti, 4)                                    # 80,000 pairs: the pinned path
    assert len(big_u) >= 1 << 16
    big = est.PredictBatch(big_u, big_i)
    assert bits_equal(big, np.tile(small, 4))
    del big, arr
    assert L.rs_knn_trim_cache() == 0


# ---- the longest rows of the exact sparse Fit: their ratings leave the CSR the column walk reads and every pair with
# one of them comes from the dense items of sim_stream_kernel (lane = popular column, register accumulators).  Every
# row (min 0: the 512 longest become popular columns) and a mix (rows of >= 150 entries), both triangles, all
# similarities; 256-column chunks, the kernels of the ML-20M shape (ML-100K defaults to 128) ----
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("pop_min", ["0", "150"])
@pytest.mark.parametrize("tri", ["upper", "lower"])
@pytest.mark.parametrize("sim", ["cosine", "msd", "pearson"])
def test_popular_columns_bit_exact(ml100k, sim, tri, pop_min, user_based, monkeypatch):
    monkeypatch.setenv("RS_KNN_STREAM_TRI", tri)
    monkeypatch.setenv("RS_KNN_STREAM_JC", "256")
    monkeypatch.setenv("RS_KNN_POP_MIN", pop_min)
    est, ref = fit_pair(ml100k["u2_base"], sim, "basic", user_based, extra={"simPath": "stream"})
    got, want = est.Sims, ref.sims()
    assert np.isnan(np.diag(got)).all()
    assert bits_equal(got, want)
    assert bits_equal(got, got.T)


# ---- popular columns with the other table type and the other similarities: continuous ratings (the dense table
# holds the b-side doubles instead of one byte per cell), PearsonBaseline with and without shrinkage (the b-side
# term depends on both biases), a threshold that makes EVERY row popular (no column walk at all), and the
# predictions that read the mirrored cells ----
@pytest.mark.parametrize("pop_min", ["0", "60"])
def test_popular_columns_tables_and_baseline(ml100k, pop_min, monkeypatch):
    monkeypatch.setenv("RS_KNN_POP_MIN", pop_min)
    arr = ml100k["u3_base"]
    u, i, r = split(arr)
    rng = np.random.RandomState(11)
    rc = r + rng.uniform(-0.49, 0.49, len(r))
    for sim in ("cosine", "msd", "pearson"):
        for user_based in (True, False):
            ts = rs.NewTrainSet(rs.NewRawSet(u, i, rc))
            est = rs.NewKNN(rs.Parameters({"sim": SIMS[sim], "userBased": user_based, "k": 40}))
            est.Fit(ts)
            ref = ob.KNN(sim=sim, knn_type="basic", user_based=user_based, k=40, n_jobs=8,
                         tie_policy="canonical").fit(ob.TrainSet(u, i, rc))
            assert bits_equal(est.Sims, ref.sims()), (sim, user_based)
    tu, ti, _ = split(ml100k["u3_test"][:3000])
    for ratings in (r, rc):
        ts = rs.NewTrainSet(rs.NewRawSet(u, i, ratings))
        ots = ob.TrainSet(u, i, ratings)
        for shrink in (0.0, 100.0):
            est = rs.NewKNNBaseLine(rs.Parameters({"sim": rs.PearsonBaseline, "userBased": False, "shrinkage": shrink}))
            est.Fit(ts)
            ref = ob.KNN(sim="pearson_baseline", knn_type="baseline", user_based=False, n_jobs=8,
                         shrinkage=shrink).fit(ots)
            assert bits_equal(est.Sims, ref.sims()), shrink
            assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti))
    # a matrix of fewer rows than the popular list can hold: every row is a popular column
    sub = arr[arr[:, 1] <= 300]
    su, si, sr = split(sub)
    est = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False, "k": 40}))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(su, si, sr)))
    ref = ob.KNN(sim="pearson", knn_type="centered", user_based=False, k=40, n_jobs=8,
                 tie_policy="canonical").fit(ob.TrainSet(su, si, sr))
    assert bits_equal(est.Sims, ref.sims())


# ---- arbitrary float64 ratings (continuous values, thousands of distinct ones): the stream path
# reads the values themselves, so anything the reference accepts is fitted (core/sim.go has no
# notion of a rating scale) ----
@pytest.mark.parametrize("knn_type", ["basic", "zscore"])
@pytest.mark.parametrize("sim", ["cosine", "msd", "pearson"])
def test_continuous_ratings_bit_exact(ml100k, sim, knn_type):
    arr = ml100k["u5_base"].copy()
    rng = np.random.RandomState(7)
    u, i, r = split(arr)
    r = r + rng.uniform(-0.49, 0.49, len(r))          # 80,000 distinct doubles
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    est = CTORS[knn_type](rs.Parameters({"sim": SIMS[sim], "userBased": True, "k": 40}))
    est.Fit(ts)
    ref = ob.KNN(sim=sim, knn_type=knn_type, user_based=True, k=40, n_jobs=8,
                 tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    assert bits_equal(est.Sims, ref.sims())
    tu, ti, _ = split(ml100k["u5_test"])
    assert bits_equal(rs.NewRawSet(tu, ti, np.zeros(len(tu))).Predict(est), ref.predict_batch(tu, ti, n_threads=8))


# ---- both chunk widths of the stream kernel (128 for small matrices, 256 for large ones); any other request
# ("512") takes 256 ----
@pytest.mark.parametrize("jc", ["128", "256", "512"])
@pytest.mark.parametrize("sim", ["cosine", "msd", "pearson"])
def test_sims_bit_exact_both_chunk_widths(ml100k, sim, jc, monkeypatch):
    monkeypatch.setenv("RS_KNN_STREAM_JC", jc)
    est, ref = fit_pair(ml100k["u3_base"], sim, "basic", False, extra={"simPath": "stream"})
    got, want = est.Sims, ref.sims()
    assert np.isnan(np.diag(got)).all()
    assert bits_equal(got, want)
    # a row shard takes the non-symmetric code path (whole runs, diagonal skipped by index)
    n = got.shape[0]
    b, e = n // 3, n // 3 + 200
    part = rs.NewKNN(rs.Parameters({"sim": SIMS[sim], "userBased": False, "simPath": "stream",
                                    "rowBegin": b, "rowEnd": e}))
    u, i, r = split(ml100k["u3_base"])
    part.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    assert bits_equal(part.Sims, want[b:e])


# ---- Predict: 4 KNN types, default config of the reference's tests (user-based MSD k=40) ----
@pytest.mark.parametrize("knn_type", ["basic", "centered", "zscore", "baseline"])
def test_predict_bit_exact_default_config(ml100k, knn_type):
    est, ref = fit_pair(ml100k["u1_base"], "msd", knn_type, True, extra={"simPath": "stream"})
    u, i, r = split(ml100k["u1_test"])
    got = rs.NewRawSet(u, i, r).Predict(est)
    want = ref.predict_batch(u, i, n_threads=8)
    assert bits_equal(got, want)
    if knn_type in ("centered", "zscore"):
        assert bits_equal(est.Means, ref.means())
    if knn_type == "zscore":
        assert bits_equal(est.StdDevs, ref.stddevs())
    # the reference's own acceptance bound for this configuration (core/base_test.go:50-64),
    # on the fixed fold u1 (harder than random folds, and its sorted row order hurts the SGD baseline)
    bound = {"basic": 0.980, "centered": 0.951, "zscore": 0.951, "baseline": 0.931}[knn_type]
    fin = np.isfinite(got)
    assert rs.RMSE(got[fin], r[fin]) <= bound + 0.03


@pytest.mark.parametrize("sim,knn_type,user_based,k", [("pearson", "centered", False, 40),
                                                        ("cosine", "basic", True, 40),
                                                        ("pearson", "zscore", True, 10),
                                                        ("cosine", "baseline", False, 100)])
def test_predict_bit_exact_other_configs(ml100k, sim, knn_type, user_based, k):
    est, ref = fit_pair(ml100k["u2_base"], sim, knn_type, user_based, k=k, extra={"simPath": "stream"})
    u, i, r = split(ml100k["u2_test"])
    got = rs.NewRawSet(u, i, r).Predict(est)
    want = ref.predict_batch(u, i, n_threads=8)
    # negative similarities are kept and nothing is clipped (core/knn.go:95-131): +-Inf / NaN and
    # out-of-range values must be reproduced, not "fixed"
    assert bits_equal(got, want)


def test_neighbour_indices_bit_exact(ml100k):
    est, ref = fit_pair(ml100k["u1_base"], "pearson", "centered", False)
    u, i, _ = split(ml100k["u1_test"])
    rng = np.random.RandomState(0)
    for x in rng.choice(len(u), 300, replace=False):
        gi, gs = est.Neighbors(int(u[x]), int(i[x]))
        wi, ws = ref.predict_neighbors(int(u[x]), int(i[x]))
        assert np.array_equal(gi.astype(np.int64), wi), x
        assert bits_equal(gs, ws)


def test_single_predict_equals_batch(ml100k):
    est, _ = fit_pair(ml100k["u1_base"][:30000], "msd", "basic", True)
    u, i, r = split(ml100k["u1_test"][:50])
    batch = est.PredictBatch(u, i)
    for x in range(50):
        assert bits_equal([est.Predict(int(u[x]), int(i[x]))], [batch[x]])


def test_cold_start_and_mink(ml100k):
    est, ref = fit_pair(ml100k["u1_base"][:20000], "msd", "basic", True, mink=5)
    u, i, _ = split(ml100k["u1_test"])
    got = est.PredictBatch(u, i)
    want = ref.predict_batch(u, i)
    assert bits_equal(got, want)
    assert (got == est.GlobalMean).sum() > 100                       # cold start + `<= mink` branch
    assert est.Predict(10 ** 9, int(i[0])) == est.GlobalMean         # newID, core/knn.go:89-91
    assert est.Predict(int(u[0]), 10 ** 9) == est.GlobalMean


def test_topk_rows(ml100k):
    est, ref = fit_pair(ml100k["u1_base"], "cosine", "basic", True)
    for k in (1, 40, 100):
        gi, gs = est.TopK(k)
        wi, ws = ref.topk(k)
        assert np.array_equal(gi, wi)
        assert bits_equal(gs, ws)


def topk_only_vs_matrix(ml100k, base, rows=None):
    """The lists of an RS_STORE_TOPK handle (k = 100) against rs_knn_topk of the matrix handle, bit for bit; with
    `rows`, a rowBegin/rowEnd top-k handle against those rows of the matrix."""
    u, i, r = split(ml100k["u1_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    full = rs.NewKNN(rs.Parameters(base))
    full.Fit(ts)
    extra = {"rowBegin": rows[0], "rowEnd": rows[1]} if rows else {}
    only = rs.NewKNN(rs.Parameters(dict(base, store="topk", topk=100, **extra)))
    only.Fit(ts)
    a, b = full.TopK(100), only.TopK(100)
    if rows:
        a = (a[0][rows[0]:rows[1]], a[1][rows[0]:rows[1]])
    assert b[0].shape == a[0].shape
    assert np.array_equal(a[0], b[0]) and bits_equal(a[1], b[1])
    return only, u, i


def test_topk_only_store_matches_matrix_store(ml100k):
    only, u, i = topk_only_vs_matrix(ml100k, {"sim": rs.MSD, "userBased": True})
    with pytest.raises(rs.core.RsError):
        only.PredictBatch(u[:4], i[:4])


@pytest.mark.parametrize("path,rows", [
    ("tensor", None),                     # 943 rows -> 8 slabs
    ("stream", None),
    ("stream", (128, 768)),               # a row shard of the top-k store: 5 slabs
])
def test_topk_only_store_row_slabs(ml100k, path, rows, monkeypatch):
    """The full-row slab loop of RS_STORE_TOPK (shard_count 0) run several times: 128-row slabs."""
    monkeypatch.setenv("RS_KNN_SLAB_ROWS", "128")
    topk_only_vs_matrix(ml100k, {"sim": rs.MSD, "userBased": True, "simPath": path}, rows)


@pytest.mark.parametrize("sim,path", [("msd", "tensor"), ("cosine", "tensor"), ("msd", "stream"),
                                      ("pearson", "stream")])
def test_symmetric_slab_topk(ml100k, sim, path, monkeypatch):
    """RS_STORE_TOPK with shard_count >= 1: every pair is computed once (right of the diagonal) and
    feeds both rows' lists.  One shard = the complete lists; three shards on one GPU, united with
    rs_knn_topk_union_device, = the same lists (multi-GPU without a cluster, SURVEY.md §4.4)."""
    import torch

    from recommend_sys_b200.shard import union_topk_device

    monkeypatch.setenv("RS_KNN_SLAB_ROWS", "256")     # 943 rows -> 4 slabs
    u, i, r = split(ml100k["u2_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    k = 50
    base = {"sim": SIMS[sim], "userBased": True, "simPath": path}
    full = rs.NewKNN(rs.Parameters(base))
    full.Fit(ts)
    want_i, want_s = full.TopK(k)
    one = rs.NewKNN(rs.Parameters(dict(base, store="topk", topk=k, shardCount=1)))
    one.Fit(ts)
    got_i, got_s = one.TopK(k)
    assert np.array_equal(got_i, want_i) and bits_equal(got_s, want_s)
    parts = []
    for rank in range(3):
        p = rs.NewKNN(rs.Parameters(dict(base, store="topk", topk=k, shardCount=3, shardIndex=rank)))
        p.Fit(ts)
        parts.append(p.TopK(k))
        p.Close()
    all_i = torch.from_numpy(np.stack([a for a, _ in parts])).cuda()
    all_s = torch.from_numpy(np.stack([b for _, b in parts])).cuda()
    uni_i, uni_s = union_topk_device(all_i, all_s)
    torch.cuda.synchronize()
    assert np.array_equal(uni_i.cpu().numpy(), want_i) and bits_equal(uni_s.cpu().numpy(), want_s)


@pytest.mark.parametrize("cap", ["1792", "96"])
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd"])
def test_fused_topk_epilogue(ml100k, sim, user_based, cap, monkeypatch):
    """RS_STORE_TOPK on the tensor path with the selection FUSED into the pair kernel's epilogue (threshold
    compare -> candidate append -> merge between the bands of the tile schedule): no similarity row is ever
    stored.  Forced on the small fixture (large problems take it by themselves); cap = 96 < the band width
    drives every row through the overflow path (threshold raised, band re-run for the flagged rows)."""
    import torch

    from recommend_sys_b200.shard import union_topk_device

    monkeypatch.setenv("RS_KNN_TOPK_FUSED", "1")
    monkeypatch.setenv("RS_KNN_TOPK_CAP", cap)
    u, i, r = split(ml100k["u3_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    k = 40
    base = {"sim": SIMS[sim], "userBased": user_based, "simPath": "tensor"}
    full = rs.NewKNN(rs.Parameters(dict(base, simPath="stream")))
    full.Fit(ts)
    want_i, want_s = full.TopK(k)
    one = rs.NewKNN(rs.Parameters(dict(base, store="topk", topk=k, shardCount=1)))
    one.Fit(ts)
    got_i, got_s = one.TopK(k)
    assert np.array_equal(got_i, want_i) and bits_equal(got_s, want_s)
    parts = []
    for rank in range(3):
        p = rs.NewKNN(rs.Parameters(dict(base, store="topk", topk=k, shardCount=3, shardIndex=rank)))
        p.Fit(ts)
        parts.append(p.TopK(k))
        p.Close()
    all_i = torch.from_numpy(np.stack([a for a, _ in parts])).cuda()
    all_s = torch.from_numpy(np.stack([b for _, b in parts])).cuda()
    uni_i, uni_s = union_topk_device(all_i, all_s)
    torch.cuda.synchronize()
    assert np.array_equal(uni_i.cpu().numpy(), want_i) and bits_equal(uni_s.cpu().numpy(), want_s)


def test_row_shards_equal_full(ml100k):
    """Multi-GPU without a cluster (SURVEY.md §4.4): the S-shard partition on one GPU equals
    the 1-shard result."""
    from recommend_sys_b200.shard import shard_rows

    u, i, r = split(ml100k["u1_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    full = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False}))
    full.Fit(ts)
    S = full.Sims
    ti, tsim = full.TopK(40)
    tu, tit, _ = split(ml100k["u1_test"][:4000])
    want = full.PredictBatch(tu, tit)
    n = ts.ItemCount
    got = np.full(len(tu), np.nan)
    for rank in range(3):
        b, e = shard_rows(n, 3, rank)
        part = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False, "rowBegin": b, "rowEnd": e}))
        part.Fit(ts)
        assert bits_equal(part.Sims, S[b:e])
        pi, ps = part.TopK(40)
        assert np.array_equal(pi, ti[b:e]) and bits_equal(ps, tsim[b:e])
        mine = (ts.convert_items(tit) >= b) & (ts.convert_items(tit) < e)
        got[mine] = part.PredictBatch(tu[mine], tit[mine])
    unknown = ts.convert_items(tit) < 0
    got[unknown] = full.GlobalMean
    assert bits_equal(got, want)


def test_non_integer_ratings_table_class(ml100k):
    """Half-star style ratings (not representable as small integers): the stream path works on
    a value table and must still be bit-exact."""
    arr = ml100k["u1_base"][:40000]
    u, i, r = split(arr)
    r = r - 0.5 * ((u + i) % 2)          # 0.5 .. 5.0 in half steps
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    ots = ob.TrainSet(u, i, r)
    for sim in ("cosine", "msd", "pearson"):
        est = rs.NewKNNWithMean(rs.Parameters({"sim": SIMS[sim], "userBased": True}))
        est.Fit(ts)
        ref = ob.KNN(sim=sim, knn_type="centered", user_based=True, n_jobs=8).fit(ots)
        assert bits_equal(est.Sims, ref.sims())
        tu, ti, _ = split(ml100k["u1_test"][:3000])
        assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti))
        assert est.Profile()["sim_path_used"] == rs.core.RS_SIM_PATH["stream"]


def test_pearson_baseline_extension(ml100k):
    """PearsonBaseline is NOT in the reference (SURVEY.md §8 a6): parity unpinned, own oracle."""
    arr = ml100k["u1_base"][:40000]
    u, i, r = split(arr)
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    ots = ob.TrainSet(u, i, r)
    for shrink in (0.0, 100.0):
        est = rs.NewKNNBaseLine(rs.Parameters({"sim": rs.PearsonBaseline, "userBased": False, "shrinkage": shrink}))
        est.Fit(ts)
        ref = ob.KNN(sim="pearson_baseline", knn_type="baseline", user_based=False, n_jobs=8,
                     shrinkage=shrink).fit(ots)
        assert bits_equal(est.Sims, ref.sims())
        tu, ti, _ = split(ml100k["u1_test"][:3000])
        assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti))


def test_als_baselines_extension(ml100k):
    """EXTENSION, parity unpinned (no ALS in the reference): device ALS baselines are bit-identical to
    the oracle's restatement, and KNNBaseline + PearsonBaseline built on them match end to end."""
    u, i, r = split(ml100k["u4_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    bl = rs.NewBaseLine(rs.Parameters({"baseline": "als"}))
    bl.Fit(ts)
    ots = ob.TrainSet(u, i, r)
    ub, ib, mu = ots.baseline_als()
    assert bits_equal(bl.userBias, ub) and bits_equal(bl.itemBias, ib) and bl.globalBias == mu
    # non-default hyper-parameters
    bl2 = rs.NewBaseLine(rs.Parameters({"baseline": "als", "regU": 3.0, "regI": 7.5, "nEpochs": 4}))
    bl2.Fit(ts)
    ub2, ib2, _ = ots.baseline_als(reg_u=3.0, reg_i=7.5, n_epochs=4)
    assert bits_equal(bl2.userBias, ub2) and bits_equal(bl2.itemBias, ib2)
    est = rs.NewKNNBaseLine(rs.Parameters({"sim": rs.PearsonBaseline, "userBased": False, "baseline": "als",
                                           "shrinkage": 100.0}))
    est.Fit(ts)
    ref = ob.KNN(sim="pearson_baseline", knn_type="baseline", user_based=False, n_jobs=8, baseline="als",
                 shrinkage=100.0).fit(ob.TrainSet(u, i, r))
    assert bits_equal(est.Sims, ref.sims())
    tu, ti, _ = split(ml100k["u4_test"])
    assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti, n_threads=8))
    with pytest.raises(rs.core.RsError):
        rs.core._check(rs.core.knn_lib().rs_baseline_als(-1, None, None, None, 0, 1, 1, 0.0, 1.0, 1.0, 1, None, None))


@pytest.mark.parametrize("pair", ["0", "1"])
@pytest.mark.parametrize("fold", ["u1", "u5"])
def test_slope_one_bit_exact(ml100k, fold, pair, monkeypatch):
    """SURVEY.md §8 f-2 — core/slope_one.go on the device: the deviation matrix (integer co-rating
    sums on the tensor cores) and SlopeOne.Predict, bit-identical to the restated reference, signed
    zeros included; the reference's own acceptance bound (core/base_test.go:46-48) on the fold."""
    monkeypatch.setenv("RS_KNN_TC_PAIR", pair)      # single-CTA / cta_group::2 pair kernel
    u, i, r = split(ml100k[fold + "_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    est = rs.NewSlopeOne(None)
    est.Fit(ts)
    ref = ob.SlopeOne().fit(ob.TrainSet(u, i, r))
    got, want = est.dev, ref.dev()
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))       # bit for bit, -0.0 vs +0.0 too
    tu, ti, tr_ = split(ml100k[fold + "_test"])
    tu = np.concatenate([tu, [10 ** 9, tu[0], 10 ** 9]])                     # unknown user / item / both
    ti = np.concatenate([ti, [ti[0], 10 ** 9, 10 ** 9]])
    pg = rs.NewRawSet(tu, ti, np.zeros(len(tu))).Predict(est)
    pw = ref.predict_batch(tu, ti)
    assert bits_equal(pg, pw)
    assert est.Predict(int(tu[5]), int(ti[5])) == pw[5]
    assert rs.RMSE(pg[:len(tr_)], tr_) <= 0.946 + 0.03
    # a row shard equals the full matrix's rows
    n = got.shape[0]
    part = rs.NewSlopeOne(rs.Parameters({"rowBegin": 256, "rowEnd": 640}))
    part.Fit(ts)
    assert np.array_equal(part.dev.view(np.uint64), want[256:640].view(np.uint64))
    # non-integer ratings are refused loudly (tensor path only)
    with pytest.raises(rs.core.RsError):
        rs.NewSlopeOne(None).Fit(rs.NewTrainSet(rs.NewRawSet(u[:1000], i[:1000], r[:1000] + 0.5)))


def test_errors_are_loud():
    left = np.array([0, 0, 1], dtype=np.int32)
    right = np.array([0, 0, 1], dtype=np.int32)
    h = rs.core._Handle()
    with pytest.raises(rs.core.RsError) as e:      # duplicate (left,right)
        h.fit(left, right, np.array([1.0, 2.0, 3.0]), 2, 2, 2.0)
    assert e.value.code == -5
    with pytest.raises(rs.core.RsError) as e:      # id out of range
        h.fit(np.array([0, 5], dtype=np.int32), np.array([0, 1], dtype=np.int32), np.array([1.0, 2.0]), 2, 2, 1.5)
    assert e.value.code == -1
    with pytest.raises(rs.core.RsError):           # Predict before Fit
        h.predict_batch(left, right)
    with pytest.raises(rs.core.RsError) as e:      # the tensor path needs small integer ratings
        rs.core._Handle(sim="cosine", sim_path="tensor").fit(left[1:], right[1:], np.array([1.5, 2.25]), 2, 2, 1.9)
    assert e.value.code == -3
    with pytest.raises(rs.core.RsError):           # baseline KNN without bias
        rs.core._Handle(knn_type="baseline").fit(left[1:], right[1:], np.array([1.0, 2.0]), 2, 2, 1.5)
    h.close()


def test_ragged_and_tiny_inputs():
    # one rating only; rows with a single entry; an item nobody else rated
    u = np.array([5, 5, 7, 9, 9, 9], dtype=np.int64)
    i = np.array([1, 2, 2, 1, 2, 3], dtype=np.int64)
    r = np.array([3.0, 4.0, 5.0, 1.0, 2.0, 5.0])
    for user_based in (True, False):
        for sim in ("cosine", "msd", "pearson"):
            ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
            est = rs.NewKNN(rs.Parameters({"sim": SIMS[sim], "userBased": user_based, "mink": 0}))
            est.Fit(ts)
            ref = ob.KNN(sim=sim, user_based=user_based, min_k=0).fit(ob.TrainSet(u, i, r))
            assert bits_equal(est.Sims, ref.sims())
            uu, ii = np.array([5, 7, 9, 5, 11]), np.array([3, 1, 2, 1, 1])
            assert bits_equal(est.PredictBatch(uu, ii), ref.predict_batch(uu, ii))
    one = rs.NewTrainSet(rs.NewRawSet([1], [1], [4.0]))
    est = rs.NewKNN(None)
    est.Fit(one)
    assert np.isnan(est.Sims).all() and est.Predict(1, 1) == 4.0


def test_refit_is_idempotent_and_handles_are_independent(ml100k):
    u, i, r = split(ml100k["u3_base"][:30000])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    a = rs.NewKNN(rs.Parameters({"sim": rs.Cosine}))
    b = rs.NewKNN(rs.Parameters({"sim": rs.MSD}))
    a.Fit(ts)
    b.Fit(ts)
    s1 = a.Sims
    a.Fit(ts)
    assert bits_equal(a.Sims, s1)
    assert not bits_equal(b.Sims, s1)


def test_cross_validate_bounds(ml100k):
    """core/base_test.go:50-52 TestKNN through the mirrored CrossValidate: params=nil -> user-based
    MSD k=40; mean RMSE <= 0.98+0.008, MAE <= 0.774+0.008."""
    d = rs.NewRawSet(*split(ml100k["u_data"]))
    res = rs.CrossValidate(rs.NewKNN(None), d, [rs.RMSE, rs.MAE], 5, 0, None)
    assert np.mean(res[0].Tests) <= 0.98 + 0.008
    assert np.mean(res[1].Tests) <= 0.774 + 0.008


# ---- full-size, size-independent properties at the BASELINE.json config-2 shape ----
def test_ml1m_shape_properties():
    d = rs.core.synth_ratings(6040, 3706, 1_000_000, 0x5EED0002)
    n_test = 200_000
    train = rs.NewTrainSet(d.SubSet(np.arange(n_test, d.Length())))
    test = d.SubSet(np.arange(n_test))
    est = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False, "k": 40}))
    est.Fit(train)
    S = est.Sims
    assert S.shape == (train.ItemCount, train.ItemCount)
    assert np.isnan(np.diag(S)).all() and bits_equal(S, S.T)
    fin = S[np.isfinite(S)]
    assert fin.min() >= -1.0000001 and fin.max() <= 1.0000001
    # oracle on a slab of rows (the oracle finishes 256 rows x all N in seconds)
    ots = ob.TrainSet(train.Users, train.Items, train.Ratings)
    ref = ob.KNN(sim="pearson", knn_type="centered", user_based=False, n_jobs=8).fit(ots, rows=(1000, 1256))
    assert bits_equal(S[1000:1256], ref.sims()[1000:1256])
    pred = test.Predict(est)
    assert len(pred) == n_test
    # predictions of rows inside the slab are checkable against the oracle
    ii = train.convert_items(test.Items)
    sel = np.where((ii >= 1000) & (ii < 1256))[0][:2000]
    want = ref.predict_batch(test.Users[sel], test.Items[sel], n_threads=8)
    assert bits_equal(pred[sel], want)


def test_ml20m_shape_config3_and_cyclic_shards():
    """Full MovieLens-20M shape, the two gaps of the round-1 review: (a) BASELINE.json configs[2] —
    KNNBaseline over PearsonBaseline similarities with ALS baselines — similarities AND predictions against
    an oracle slab; (b) the multi-GPU form of the north-star workload — cyclic row shards, 2 and 3 shards on
    one GPU, peer mirror — equal to the unsharded matrix and predictions."""
    d = rs.core.synth_ratings(138_493, 26_744, 20_400_000, 0x5EED0003)
    n_test = 400_000
    train = rs.NewTrainSet(d.SubSet(np.arange(n_test, d.Length())))
    test = d.SubSet(np.arange(n_test))
    n = train.ItemCount
    # ---- (a) config 3 ----
    est = rs.NewKNNBaseLine(rs.Parameters({"sim": rs.PearsonBaseline, "userBased": False, "k": 40, "baseline": "als"}))
    est.Fit(train)
    r0, r1 = 9000, 9040
    ots = ob.TrainSet(train.Users, train.Items, train.Ratings)
    ref = ob.KNN(sim="pearson_baseline", knn_type="baseline", user_based=False, k=40, n_jobs=16,
                 baseline="als").fit(ots, rows=(r0, r1))
    assert bits_equal(est._h.sims_rows(r0, r1 - r0), ref.sims(copy=False)[r0:r1])
    ii = train.convert_items(test.Items)
    sel = np.where((ii >= r0) & (ii < r1))[0][:400]
    assert len(sel) > 50
    assert bits_equal(est.PredictBatch(test.Users[sel], test.Items[sel]),
                      ref.predict_batch(test.Users[sel], test.Items[sel], n_threads=16))
    est.Close()
    del ref
    # ---- (b) cyclic row shards of the north-star workload ----
    base = {"sim": rs.Pearson, "userBased": False, "k": 40}
    full = rs.NewKNNWithMean(rs.Parameters(base))
    full.Fit(train)
    want_pred = test.Predict(full)
    probe = [0, 32, 4992, 13344, 26720]                          # block starts across the matrix
    want_rows = {b: full._h.sims_rows(b, min(32, n - b)) for b in probe}
    full.Close()
    left = train.convert_items(test.Items)
    for count in (2, 3):
        shards = []
        for q in range(count):
            e = rs.NewKNNWithMean(rs.Parameters(dict(base, shardCount=count, shardIndex=q)))
            e.Fit(train)
            shards.append(e)
        for e in shards:
            e._h.synchronize()
        for e in shards:
            e._h.peer_import_local([x._h for x in shards])
            e._h.mirror()
        owner = rs.shard.route_pairs(left, count)
        got = np.full(n_test, np.nan)
        for q, e in enumerate(shards):
            mine = np.flatnonzero(owner == q)
            got[mine] = e.PredictBatch(test.Users[mine], test.Items[mine])
            for b in probe:
                if rs.core.cyclic_owner(b, count) == q:
                    assert bits_equal(e._h.sims_rows(b, min(32, n - b)), want_rows[b]), (count, q, b)
        assert bits_equal(got, want_pred), count
        for e in shards:
            e.Close()


def test_ml20m_shape_properties():
    """BASELINE.json's target shape (item-based Pearson, k=40, MovieLens-20M: 138,493 x 26,744, 20 M
    ratings) at FULL size: size-independent properties of the 5.7 GB similarity matrix checked on
    slabs, plus an oracle slab of 48 rows x all N and the predictions that fall inside it."""
    d = rs.core.synth_ratings(138_493, 26_744, 20_400_000, 0x5EED0003)
    n_test = 400_000
    train = rs.NewTrainSet(d.SubSet(np.arange(n_test, d.Length())))
    test = d.SubSet(np.arange(n_test))
    est = rs.NewKNNWithMean(rs.Parameters({"sim": rs.Pearson, "userBased": False, "k": 40}))
    est.Fit(train)
    n = train.ItemCount
    h = est._h
    a0, b0, m = 5000, 20000, 512
    A = h.sims_rows(a0, m)
    B = h.sims_rows(b0, m)
    assert A.shape == (m, n)
    assert np.isnan(A[np.arange(m), a0 + np.arange(m)]).all()             # diagonal unset (core/knn.go:202)
    assert bits_equal(A[:, b0:b0 + m], B[:, a0:a0 + m].T)                 # Sims[i][j] == Sims[j][i] (core/knn.go:205-208)
    assert bits_equal(A[:, a0:a0 + m], A[:, a0:a0 + m].T)
    fin = A[np.isfinite(A)]
    assert fin.min() >= -1.0000001 and fin.max() <= 1.0000001
    # oracle slab (rows r0..r0+48 x all N)
    r0, r1 = 5000, 5048
    ots = ob.TrainSet(train.Users, train.Items, train.Ratings)
    ref = ob.KNN(sim="pearson", knn_type="centered", user_based=False, n_jobs=16).fit(ots, rows=(r0, r1))
    want = ref.sims(copy=False)[r0:r1]
    assert bits_equal(A[r0 - a0:r1 - a0], want)
    pred = test.Predict(est)
    assert len(pred) == n_test
    ii = train.convert_items(test.Items)
    sel = np.where((ii >= r0) & (ii < r1))[0][:500]
    assert len(sel) > 50
    assert bits_equal(pred[sel], ref.predict_batch(test.Users[sel], test.Items[sel], n_threads=16))
    del ref
    # the popular rows (first-appearance ids: the blockbusters are among the first rows): their pairs come from
    # the dense pass and the mirror, not from the column walk — an oracle slab over them, and their transposes
    cnt_items = np.bincount(train.innerItems, minlength=n)
    assert (cnt_items[:256] >= 8192).sum() >= 8               # the slab below does hold popular rows
    P0 = h.sims_rows(0, 256)
    refp = ob.KNN(sim="pearson", knn_type="centered", user_based=False, n_jobs=16).fit(ots, rows=(0, 12))
    assert bits_equal(P0[:12], refp.sims(copy=False)[0:12])
    del refp
    assert np.isnan(P0[np.arange(256), np.arange(256)]).all()
    assert bits_equal(P0[:, :256], P0[:, :256].T)
    assert bits_equal(P0[:, a0:a0 + m], A[:, :256].T)
    assert bits_equal(P0[:, b0:b0 + m], B[:, :256].T)
    # the dense tensor path agrees bit for bit with the sparse replay on Cosine at this size
    cos_t = rs.NewKNN(rs.Parameters({"sim": rs.Cosine, "userBased": False, "simPath": "tensor"}))
    cos_t.Fit(train)
    T1 = cos_t._h.sims_rows(a0, 256)
    cos_t.Close()
    cos_s = rs.NewKNN(rs.Parameters({"sim": rs.Cosine, "userBased": False, "simPath": "stream"}))
    cos_s.Fit(train)
    assert bits_equal(T1, cos_s._h.sims_rows(a0, 256))
    cos_s.Close()
    est.Close()
    # Pearson from the six integer sums on the tensor cores (K = 138 k) against the exact replay
    ps = rs.NewKNN(rs.Parameters({"sim": rs.Pearson, "userBased": False, "pearsonMode": "sums", "simPath": "tensor"}))
    ps.Fit(train)
    assert ps.Profile()["sim_path_used"] == rs.core.RS_SIM_PATH["tensor"]
    P = ps._h.sims_rows(a0, m)
    ps.Close()
    assert np.array_equal(np.isnan(P), np.isnan(A))
    okp = ~np.isnan(A)
    assert (np.abs(P[okp] - A[okp]) <= 1e-9 * np.maximum(1.0, np.abs(A[okp]))).all()
    # ALS baselines (extension) at full size: device == oracle bit for bit
    bl = rs.NewBaseLine(rs.Parameters({"baseline": "als"}))
    bl.Fit(train)
    oub, oib, _ = ob.TrainSet(train.Users, train.Items, train.Ratings).baseline_als()
    assert bits_equal(bl.userBias, oub) and bits_equal(bl.itemBias, oib)
    # Slope One (SURVEY.md §8 f-2) at full size: cells against a direct evaluation of core/slope_one.go:74-88
    so = rs.NewSlopeOne(None)
    so.Fit(train)
    D = so._h.sims_rows(a0, 64)
    by_item = {}
    iu, ii, rr = train.innerUsers, train.innerItems, train.Ratings
    rng = np.random.RandomState(3)
    pairs = [(a0 + int(x), int(y)) for x, y in zip(rng.randint(0, 64, 40), rng.randint(0, n, 40))] + [(a0 + 3, a0 + 3)]
    for i_, j_ in pairs:
        for t_ in (i_, j_):
            if t_ not in by_item:
                sel = np.where(ii == t_)[0]
                by_item[t_] = dict(zip(iu[sel].tolist(), rr[sel].tolist()))
        common = sorted(set(by_item[i_]) & set(by_item[j_]))
        if i_ == j_ or not common:
            want = 0.0
        else:
            big, small = max(i_, j_), min(i_, j_)
            ssum = 0.0
            for u_ in common:                       # ascending user id, as the merge walks them
                ssum += by_item[big][u_] - by_item[small][u_]
            want = ssum / float(len(common))
            if i_ < j_:
                want = -want
        assert D[i_ - a0, j_] == want and np.signbit(D[i_ - a0, j_]) == np.signbit(want), (i_, j_)
    E_ = so._h.sims_rows(b0, 64)
    assert np.array_equal(D[:, b0:b0 + 64], -E_[:, a0:a0 + 64].T + 0.0) or \
        np.array_equal(np.abs(D[:, b0:b0 + 64]), np.abs(E_[:, a0:a0 + 64].T))       # antisymmetric
    # SlopeOne.Predict for pairs whose item row is in the slab: sequential sum in dataset order
    tu = train.convert_users(test.Users)
    ti = train.convert_items(test.Items)
    sel = np.where((ti >= a0) & (ti < a0 + 64) & (tu >= 0))[0][:40]
    got = so.PredictBatch(test.Users[sel], test.Items[sel])
    cnt = np.bincount(iu, minlength=train.UserCount)
    for x, q in enumerate(sel):
        rows_u = np.where(iu == tu[q])[0]                               # dataset order
        ssum = 0.0
        for it_ in ii[rows_u]:
            ssum += D[ti[q] - a0, it_]
        want = float(np.add.reduce(rr[rows_u]) / len(rows_u)) + ssum / float(len(rows_u))
        assert got[x] == want, (q, got[x], want)
    so.Close()


def test_config4_shape_symmetric_slab_topk():
    """BASELINE.json config 4 at FULL size: user-based MSD, k = 100, MovieLens-20M shape (138,493 users,
    9.6e9 pairs; the 153 GB matrix never exists).  Neighbour lists from the symmetric-slab Fit — one
    shard, and two shards on one GPU united with rs_knn_topk_union_device — against rows computed by
    the oracle straight from core/sim.go: indices and similarities bit for bit."""
    import torch

    from recommend_sys_b200.shard import union_topk_device

    d = rs.core.synth_ratings(138_493, 26_744, 20_000_000, 0x5EED0004)
    train = rs.NewTrainSet(d)
    n, k = train.UserCount, 100
    base = {"sim": rs.MSD, "userBased": True, "store": "topk", "topk": k}
    one = rs.NewKNN(rs.Parameters(dict(base, shardCount=1)))
    one.Fit(train)
    gi, gs = one.TopK(k)
    one.Close()
    assert gi.shape == (n, k)
    rows = np.array([0, 1, 777, 5000, 65535, 65536, 100_000, n - 2, n - 1], dtype=np.int64)
    S = ob.rows_sims(ob.TrainSet(train.Users, train.Items, train.Ratings), "msd", True, rows)
    for x, row in enumerate(rows):
        s = S[x]
        ok = np.where(~np.isnan(s))[0]
        order = ok[np.lexsort((ok, -s[ok]))][:k]                      # similarity desc, inner id asc
        assert np.array_equal(gi[row][:len(order)], order), row
        assert bits_equal(gs[row][:len(order)], s[order]), row
        assert (gi[row][len(order):] == -1).all()
    parts = []
    for rank in range(2):
        p = rs.NewKNN(rs.Parameters(dict(base, shardCount=2, shardIndex=rank)))
        p.Fit(train)
        parts.append(p.TopK(k))
        p.Close()
    ui, us = union_topk_device(torch.from_numpy(np.stack([a for a, _ in parts])).cuda(),
                               torch.from_numpy(np.stack([b for _, b in parts])).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(ui.cpu().numpy(), gi) and bits_equal(us.cpu().numpy(), gs)



def test_netflix_shape_tensor_stream_oracle():
    """BASELINE.json config 5 at FULL size (item-based Cosine on the Netflix-Prize shape: 480,189 users x
    17,770 items, 100 M ratings; K = 480 k is the longest contraction of any config): the CTA-pair tensor
    kernel and the exact sparse replay agree bit for bit on a slab, and both agree with oracle rows
    straight from core/sim.go."""
    d = rs.core.synth_ratings(480_189, 17_770, 100_000_000, 0x5EED0005)
    train = rs.NewTrainSet(d)
    n = train.ItemCount
    a = rs.NewKNN(rs.Parameters({"sim": rs.Cosine, "userBased": False, "simPath": "tensor", "k": 50}))
    a.Fit(train)
    assert a.Profile()["sim_path_used"] == rs.core.RS_SIM_PATH["tensor"]
    T = a._h.sims_rows(3000, 256)
    T2 = a._h.sims_rows(n - 200, 200)
    # KNN.Predict (k = 50) for item 3000 and users of very different activity, restated here from
    # core/knn.go:75-141 on the device's own similarity row (canonical tie rule)
    iu, ii, rr = train.innerUsers, train.innerItems, train.Ratings
    deg = np.bincount(iu, minlength=train.UserCount)
    users = [int(np.argmax(deg)), int(np.argsort(deg)[len(deg) // 2]), int(np.argmin(deg)), 12345, 400_000]
    raw_item = int(train.Items[np.where(ii == 3000)[0][0]])
    raw_users = [int(train.Users[np.where(iu == u_)[0][0]]) for u_ in users]
    got = a.PredictBatch(np.array(raw_users), np.array([raw_item] * len(users)))
    for x, u_ in enumerate(users):
        sel = np.where(iu == u_)[0]
        ids, rat = ii[sel], rr[sel]
        sv = T[0][ids]
        ok = ~np.isnan(sv)
        if ok.sum() <= 1:
            want = train.GlobalMean
        else:
            order = np.lexsort((ids[ok], -(sv[ok] + 0.0)))[:50]
            ws = wr = 0.0
            for t_ in order:
                ws += sv[ok][t_]
                wr += sv[ok][t_] * rat[ok][t_]
            want = wr / ws
        assert got[x] == want, (u_, got[x], want)
    a.Close()
    b = rs.NewKNN(rs.Parameters({"sim": rs.Cosine, "userBased": False, "simPath": "stream"}))
    b.Fit(train)
    assert bits_equal(T, b._h.sims_rows(3000, 256))
    assert bits_equal(T2, b._h.sims_rows(n - 200, 200))
    b.Close()
    rows = np.array([3000, 3100, n - 1], dtype=np.int64)
    S = ob.rows_sims(ob.TrainSet(train.Users, train.Items, train.Ratings), "cosine", False, rows)
    assert bits_equal(T[[0, 100]], S[:2]) and bits_equal(T2[-1:], S[2:])
