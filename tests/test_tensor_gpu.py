"""Parity of the tcgen05 int8 path (sim_tensor.cu) through the C ABI.

Integer co-rating sums must be bit-exact; Cosine and MSD similarities computed from them must be
bit-identical to the oracle (their Go sums are sums of small integers, exact in float64);
Pearson in `sums` mode is held to |d| <= 1e-9 * max(1, |ref|) (SURVEY.md §7.3 item 2) with an
exactly matching NaN pattern, and to 4 ulps of the exact value of its integer sums (tests/exact_sums.py)."""
import numpy as np
import pytest

import recommend_sys_b200 as rs
from oracle import binding as ob
from conftest import bits_equal, split

pytestmark = pytest.mark.gpu

SIMS = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson}


def _fit(arr, sim, user_based, **extra):
    u, i, r = split(arr)
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    p = {"sim": SIMS[sim], "userBased": user_based, "simPath": "tensor"}
    p.update(extra)
    est = rs.NewKNN(rs.Parameters(p))
    est.Fit(ts)
    ref = ob.KNN(sim=sim, user_based=user_based, n_jobs=8).fit(ob.TrainSet(u, i, r))
    return est, ref, ts


@pytest.mark.parametrize("user_based", [True, False])
def test_cosums_bit_exact(ml100k, user_based):
    est, ref, ts = _fit(ml100k["u1_base"], "msd", user_based)
    n = ts.UserCount if user_based else ts.ItemCount
    for row0, nrows in ((0, 3), (127, 4), (n - 2, 2)):
        got = est._h.cosums(row0, nrows)
        assert got.shape == (nrows, n, 6)
        rng = np.random.RandomState(row0)
        cols = np.unique(np.concatenate([rng.choice(n, 200), [0, 63, 64, 127, 128, n - 1]]))
        for r in range(nrows):
            for c in cols:
                want = ref.pair_sums(row0 + r, int(c))
                assert np.array_equal(got[r, c].astype(np.int64), want), (row0 + r, int(c))


# kernel variants: the single-CTA kernel (small problems) and the cta_group::2 CTA-pair kernel (the default on
# large Cosine / MSD problems) — forced here on ml-100k
VARIANTS = {"single": {"RS_KNN_TC_PAIR": "0"},
            "pair": {"RS_KNN_TC_PAIR": "1"}}


@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", ["cosine", "msd"])
def test_tensor_sims_bit_exact(ml100k, sim, user_based, variant, monkeypatch):
    for k, v in VARIANTS[variant].items():
        monkeypatch.setenv(k, v)
    est, ref, _ = _fit(ml100k["u1_base"], sim, user_based)
    assert est.Profile()["sim_path_used"] == rs.core.RS_SIM_PATH["tensor"]
    got, want = est.Sims, ref.sims()
    assert np.isnan(np.diag(got)).all()
    assert bits_equal(got, want)


def test_tensor_equals_stream_path(ml100k):
    u, i, r = split(ml100k["u3_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    for sim in (rs.Cosine, rs.MSD):
        a = rs.NewKNN(rs.Parameters({"sim": sim, "simPath": "tensor"}))
        b = rs.NewKNN(rs.Parameters({"sim": sim, "simPath": "stream"}))
        a.Fit(ts)
        b.Fit(ts)
        assert bits_equal(a.Sims, b.Sims)


def test_tensor_predict_bit_exact(ml100k):
    est, ref, _ = _fit(ml100k["u2_base"], "cosine", True)
    u, i, _r = split(ml100k["u2_test"])
    assert bits_equal(est.PredictBatch(u, i), ref.predict_batch(u, i, n_threads=8))


@pytest.mark.parametrize("pair", ["0", "1"])
def test_tensor_row_shard(ml100k, pair, monkeypatch):
    from recommend_sys_b200.shard import shard_rows

    monkeypatch.setenv("RS_KNN_TC_PAIR", pair)
    u, i, r = split(ml100k["u1_base"])
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    full = rs.NewKNN(rs.Parameters({"sim": rs.MSD, "userBased": False, "simPath": "tensor"}))
    full.Fit(ts)
    S = full.Sims
    for rank in range(2):
        b, e = shard_rows(ts.ItemCount, 2, rank)
        part = rs.NewKNN(rs.Parameters({"sim": rs.MSD, "userBased": False, "simPath": "tensor", "rowBegin": b,
                                        "rowEnd": e}))
        part.Fit(ts)
        assert bits_equal(part.Sims, S[b:e])


def test_pearson_sums_mode_tolerance(ml100k):
    """Both orientations: within 1e-9 of the oracle's replay, and against the exact integer sums (tests/exact_sums.py)
    NaN exactly where Mi Ni == 0, +0.0 exactly where L == 0, bit-symmetric, within 4 ulps of the exact value."""
    import exact_sums as ex

    for user_based in (False, True):
        est, ref, ts = _fit(ml100k["u1_base"], "pearson", user_based, pearsonMode="sums")
        assert est.Profile()["sim_path_used"] == rs.core.RS_SIM_PATH["tensor"]
        got, want = est.Sims, ref.sims()
        assert np.array_equal(np.isnan(got), np.isnan(want))        # NaN-ness decided on exact integers
        ok = ~np.isnan(want)
        err = np.abs(got[ok] - want[ok])
        assert (err <= 1e-9 * np.maximum(1.0, np.abs(want[ok]))).all(), err.max()
        assert bits_equal(got, got.T)
        left, right = (ts.innerUsers, ts.innerItems) if user_based else (ts.innerItems, ts.innerUsers)
        n_left, n_right = (ts.UserCount, ts.ItemCount) if user_based else (ts.ItemCount, ts.UserCount)
        L, Mi, Ni = ex.Sums(left, right, ts.Ratings, n_left, n_right).pearson_terms()
        worst = ex.check_ratio(got, L, Mi, Ni, who=f"user_based={user_based}")
        print(f"\nML-100K Pearson sums user_based={user_based}: max ulps (<2^53, >=2^53) = {worst}")


def test_tensor_rejects_non_integer_ratings():
    left = np.array([0, 0, 1, 1], dtype=np.int32)
    right = np.array([0, 1, 0, 1], dtype=np.int32)
    h = rs.core._Handle(sim="cosine", sim_path="tensor")
    with pytest.raises(rs.core.RsError) as e:
        h.fit(left, right, np.array([1.5, 2.0, 3.0, 4.0]), 2, 2, 2.6)
    assert e.value.code == -3
    h.close()


@pytest.mark.parametrize("pair", ["0", "1"])
def test_tensor_tiny_and_odd_shapes(pair, monkeypatch):
    monkeypatch.setenv("RS_KNN_TC_PAIR", pair)
    rng = np.random.RandomState(5)
    for n_users, n_items, nnz in ((3, 5, 9), (130, 70, 2000), (257, 129, 5000)):
        cells = rng.choice(n_users * n_items, nnz, replace=False)
        u, i = cells // n_items, cells % n_items
        r = rng.randint(0, 6, nnz).astype(np.float64)        # rating 0 is a legal value (mask plane)
        for user_based in (True, False):
            for sim in ("cosine", "msd"):
                ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
                est = rs.NewKNN(rs.Parameters({"sim": SIMS[sim], "userBased": user_based, "simPath": "tensor"}))
                est.Fit(ts)
                ref = ob.KNN(sim=sim, user_based=user_based).fit(ob.TrainSet(u, i, r))
                assert bits_equal(est.Sims, ref.sims()), (n_users, n_items, sim, user_based)
