"""Host restatement of recommendation for queries given as rating lists (tests/recommend_given_ref.py), pinned to the
oracle without a GPU, and the Python grouping of KNN.ScoreAllGiven / RecommendGiven."""
import numpy as np
import pytest

from conftest import split
from recommend_given_ref import KNN_TYPES, Model, list_stats, user_lists
from recommend_ref import same_bits, score_all

SIMS = ("cosine", "msd", "pearson")
USERS = np.arange(0, 943, 37)          # 26 users of ML-100K u1, light and heavy raters


@pytest.mark.parametrize("user_based", [True, False])
@pytest.mark.parametrize("sim", SIMS)
@pytest.mark.parametrize("knn_type", KNN_TYPES)
def test_own_ratings_are_the_oracle_predictions(ml100k, sim, knn_type, user_based):
    """A list that is a fitted user's own ratings (dataset order) gives the oracle's Predict on every unrated target,
    bit for bit.  Left (user-based) queries with a baseline bias are refused by the library and not restated."""
    if user_based and knn_type == "baseline":
        pytest.skip("left queries have no baseline bias")
    u, i, r = split(ml100k["u1_base"])
    m = Model(u, i, r, sim, knn_type, user_based)
    side = "left" if user_based else "right"
    users, ptr, ids, vals = user_lists(u, i, r, USERS)
    got = m.score_all_given(side, ptr, ids, vals)
    want = score_all(m.ref, u, i, user_based, side, users)
    assert same_bits(got, want)


def test_right_side_ignores_the_list_order(ml100k):
    u, i, r = split(ml100k["u1_base"])
    m = Model(u, i, r, "pearson", "centered", False)
    _, ptr, ids, vals = user_lists(u, i, r, USERS[:5])
    rng = np.random.RandomState(1)
    for b in range(5):
        sl = slice(ptr[b], ptr[b + 1])
        p = rng.permutation(ptr[b + 1] - ptr[b])
        assert same_bits(m.score_given("right", ids[sl][p], vals[sl][p]), m.score_given("right", ids[sl], vals[sl]))


def test_empty_list_is_global_mean(ml100k):
    u, i, r = split(ml100k["u1_base"])
    for user_based in (True, False):
        m = Model(u, i, r, "msd", "centered", user_based)
        side = "left" if user_based else "right"
        row = m.score_given(side, np.empty(0, np.int64), np.empty(0))
        assert (row == m.global_mean).all()


def test_list_stats_follow_the_caller_order():
    vals = [1e16, 1.0, -1e16, 1.0]
    assert list_stats(vals)[0] == ((((1e16 + 1.0) - 1e16) + 1.0) / 4)
    assert list_stats(vals[::-1])[0] != list_stats(vals)[0]    # the order the ratings were given is the order summed


# ---- the Python mirror: grouping and raw-id mapping, no device needed ----
class _FakeHandle:
    def __init__(self):
        self.calls = []

    def score_all_given(self, side, ptr, ids, vals):
        self.calls.append(("score", side, ptr, ids, vals))
        return np.zeros((len(ptr) - 1, 4))

    def recommend_given(self, side, ptr, ids, vals, n):
        self.calls.append(("rec", side, ptr, ids, vals))
        out = np.full((len(ptr) - 1, n), -1, dtype=np.int32)
        out[:, 0] = [2, 0, 3][:len(ptr) - 1]
        return out, np.zeros((len(ptr) - 1, n))


def _knn_with_fake(user_based):
    import recommend_sys_b200 as rs

    train = rs.NewTrainSet(rs.NewRawSet(np.array([10, 10, 20, 30]), np.array([100, 200, 300, 400]),
                                        np.array([1.0, 2.0, 3.0, 4.0])))
    est = rs.NewKNN(rs.Parameters({"userBased": user_based}))
    est.Data = train
    est._userBased = user_based
    est._kk = (40, 1)
    est._h = _FakeHandle()
    return est


@pytest.mark.parametrize("user_based", [True, False])
def test_given_grouping_and_raw_ids(user_based):
    import recommend_sys_b200 as rs

    est = _knn_with_fake(user_based)
    # users 7 (new), 20 (known), 7 again, 99 (only unknown items); item 999 is unknown to the train set
    ds = rs.NewRawSet(np.array([7, 20, 7, 99, 7, 20]), np.array([300, 100, 999, 999, 100, 400]),
                      np.array([5.0, 4.0, 3.0, 2.0, 1.0, 0.5]))
    users, scores = est.ScoreAllGiven(ds)
    _, side, ptr, ids, vals = est._h.calls[-1]
    assert side == ("left" if user_based else "right")
    assert users.tolist() == [7, 20, 99]                        # order of first appearance
    assert ptr.tolist() == [0, 2, 4, 4]                          # 99 keeps an empty list
    assert ids.tolist() == [2, 0, 0, 3]                          # inner items: 100 -> 0, 300 -> 2, 400 -> 3
    assert vals.tolist() == [5.0, 1.0, 4.0, 0.5]                 # each user's entries in dataset order
    assert scores.shape == (3, 4)
    users, items, top = est.RecommendGiven(ds, 2)
    assert users.tolist() == [7, 20, 99]
    assert items[:, 0].tolist() == [300, 100, 400] and (items[:, 1] == -1).all()   # inner -> raw, -1 stays newID
    est._h = None


def test_sharded_knn_refuses_given():
    from recommend_sys_b200 import shard

    obj = shard.ShardedKNN.__new__(shard.ShardedKNN)
    with pytest.raises(NotImplementedError):
        obj.ScoreAllGiven(None)
    with pytest.raises(NotImplementedError):
        obj.RecommendGiven(None, 5)
