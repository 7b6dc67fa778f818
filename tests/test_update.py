"""TrainSet.Extend (the TrainSet KNN.Update leaves behind) against NewTrainSet of the concatenation: inner ids, counts
and GlobalMean bits, for integer and fractional ratings, with known and new ids."""
import numpy as np
import pytest

from conftest import split


def _rs():
    import recommend_sys_b200 as rs

    return rs


def _same(a, b):
    assert a.UserCount == b.UserCount and a.ItemCount == b.ItemCount
    assert np.array_equal(a.innerUsers, b.innerUsers) and np.array_equal(a.innerItems, b.innerItems)
    assert np.array_equal(a.Users, b.Users) and np.array_equal(a.Items, b.Items)
    assert np.array_equal(a.Ratings.view(np.uint64), b.Ratings.view(np.uint64))
    assert np.float64(a.GlobalMean).view(np.uint64) == np.float64(b.GlobalMean).view(np.uint64)
    for raw in (1, 5001, 9001):
        assert a.ConvertUserID(raw) == b.ConvertUserID(raw)
        assert a.ConvertItemID(raw) == b.ConvertItemID(raw)


@pytest.mark.parametrize("fractional", [False, True])
@pytest.mark.parametrize("tail", [1, 500, 8000])
def test_extend_equals_new_trainset(ml100k, fractional, tail):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    if fractional:
        r = r - 0.5 * (np.arange(len(r)) % 3 == 0) + 1e-3 * (np.arange(len(r)) % 7)
    # the tail adds known ids, and new users and items
    u = np.concatenate([u, [5001, 5001, 3]])
    i = np.concatenate([i, [1, 9001, 9001]])
    r = np.concatenate([r, [4.0, 2.5 if fractional else 2.0, 5.0]])
    m = len(r) - tail - 3
    first = rs.NewTrainSet(rs.NewRawSet(u[:m], i[:m], r[:m]))
    got = first.Extend(rs.NewRawSet(u[m:], i[m:], r[m:]))
    want = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    _same(got, want)
    assert np.array_equal(got.innerUsers[:m], first.innerUsers)       # known ids keep their inner ids
