"""TrainSet.Remove / TrainSet.Change (the TrainSets KNN.Remove and KNN.Change leave behind): inner ids and counts kept,
ids without rows still converting, Extend continuing the numbering after a removal and equal to NewTrainSet of the
concatenation on a set never edited, GlobalMean of the edited ratings, and the refusals."""
import numpy as np
import pytest

from conftest import split

RS_ERR_INVALID, RS_ERR_DUPLICATE = -1, -5


def _rs():
    import recommend_sys_b200 as rs

    return rs


def _bits(x):
    return np.float64(x).view(np.uint64)


def _train(ml100k, fractional=False):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    if fractional:
        r = r - 0.5 * (np.arange(len(r)) % 3 == 0) + 1e-3 * (np.arange(len(r)) % 7)
    return rs.NewTrainSet(rs.NewRawSet(u, i, r)), u, i, r


def _picked(n, frac, seed):
    return np.sort(np.random.RandomState(seed).choice(n, int(n * frac), replace=False))


@pytest.mark.parametrize("fractional", [False, True])
def test_remove_keeps_ids_and_counts(ml100k, fractional):
    rs = _rs()
    ts, u, i, r = _train(ml100k, fractional)
    rows = _picked(len(r), 0.1, 1)
    got = ts.Remove(u[rows][::-1], i[rows][::-1])          # the order of the pairs does not matter
    keep = np.ones(len(r), dtype=bool)
    keep[rows] = False
    assert got.UserCount == ts.UserCount and got.ItemCount == ts.ItemCount
    assert np.array_equal(got.Users, u[keep]) and np.array_equal(got.Items, i[keep])
    assert np.array_equal(got.Ratings.view(np.uint64), r[keep].view(np.uint64))
    assert np.array_equal(got.innerUsers, ts.innerUsers[keep])
    assert np.array_equal(got.innerItems, ts.innerItems[keep])
    assert _bits(got.GlobalMean) == _bits(rs.core._global_mean(r[keep]))
    for raw in np.unique(u):
        assert got.ConvertUserID(raw) == ts.ConvertUserID(raw)
    assert np.array_equal(got.convert_items(np.unique(i)), ts.convert_items(np.unique(i)))
    assert got.ConvertUserID(10 ** 6) == -1


@pytest.mark.parametrize("fractional", [False, True])
def test_change_keeps_everything_but_the_ratings(ml100k, fractional):
    rs = _rs()
    ts, u, i, r = _train(ml100k, fractional)
    rows = _picked(len(r), 0.1, 2)
    new = np.random.RandomState(3).randint(1, 6, len(rows)).astype(np.float64)
    if fractional:
        new -= 0.5
    got = ts.Change(rs.NewRawSet(u[rows], i[rows], new))
    want = r.copy()
    want[rows] = new
    assert np.array_equal(got.Ratings.view(np.uint64), want.view(np.uint64))
    assert np.array_equal(got.Users, u) and np.array_equal(got.Items, i)
    assert np.array_equal(got.innerUsers, ts.innerUsers) and np.array_equal(got.innerItems, ts.innerItems)
    assert got.UserCount == ts.UserCount and got.ItemCount == ts.ItemCount
    assert _bits(got.GlobalMean) == _bits(rs.core._global_mean(want))
    assert np.array_equal(ts.Ratings.view(np.uint64), r.view(np.uint64))   # the set itself is left as it was


def test_id_without_rows_still_converts(ml100k):
    ts, u, i, r = _train(ml100k)
    user, item = u[0], i[0]
    rows_u, rows_i = np.flatnonzero(u == user), np.flatnonzero(i == item)
    got = ts.Remove(u[rows_u], i[rows_u])
    assert user not in got.Users
    assert got.ConvertUserID(user) == ts.ConvertUserID(user) == 0
    assert got.convert_users(np.array([user]))[0] == 0
    assert got._raw_ids()[0][0] == user                  # inner -> raw, as recommendation lists map their ids
    got = got.Remove(*[a[np.isin(rows_i, rows_u, invert=True)] for a in (u[rows_i], i[rows_i])])
    assert item not in got.Items
    assert got.ConvertItemID(item) == ts.ConvertItemID(item) == 0
    assert got.UserCount == ts.UserCount and got.ItemCount == ts.ItemCount


def test_extend_after_remove_continues_the_numbering(ml100k):
    """A removal takes out the row where user u[0] and item i[0] first appeared; NewTrainSet of the remaining rows
    would renumber, Extend keeps the numbers and gives new ids the next ones."""
    rs = _rs()
    ts, u, i, r = _train(ml100k)
    first_user_rows = np.flatnonzero(u == u[0])
    removed = ts.Remove(u[first_user_rows], i[first_user_rows])
    add = rs.NewRawSet(np.array([u[0], 5001, 5002, 5001, u[5]]), np.array([i[0], 9001, i[3], i[7], 9002]),
                       np.array([4.0, 3.0, 2.0, 5.0, 1.0]))
    got = removed.Extend(add)
    assert got.UserCount == ts.UserCount + 2 and got.ItemCount == ts.ItemCount + 2
    want_u = [0, ts.UserCount, ts.UserCount + 1, ts.UserCount, ts.ConvertUserID(u[5])]
    want_i = [0, ts.ItemCount, ts.ConvertItemID(i[3]), ts.ConvertItemID(i[7]), ts.ItemCount + 1]
    assert got.innerUsers[-5:].tolist() == want_u
    assert got.innerItems[-5:].tolist() == want_i
    assert np.array_equal(got.innerUsers[:-5], removed.innerUsers)
    assert got.ConvertUserID(5002) == ts.UserCount + 1 and got.ConvertItemID(9002) == ts.ItemCount + 1
    assert _bits(got.GlobalMean) == _bits(rs.core._global_mean(np.concatenate([removed.Ratings, add.Ratings])))
    # and a removal after that still knows every id
    again = got.Remove([5002], [i[3]])
    assert again.ConvertUserID(5002) == ts.UserCount + 1 and 5002 not in again.Users


@pytest.mark.parametrize("tail", [1, 500])
def test_extend_of_an_unedited_set_equals_new_trainset(ml100k, tail):
    rs = _rs()
    u, i, r = split(ml100k["u1_base"])
    u = np.concatenate([u, [5001, 5001, 3]])
    i = np.concatenate([i, [1, 9001, 9001]])
    r = np.concatenate([r, [4.0, 2.0, 5.0]])
    m = len(r) - tail - 3
    got = rs.NewTrainSet(rs.NewRawSet(u[:m], i[:m], r[:m])).Extend(rs.NewRawSet(u[m:], i[m:], r[m:]))
    want = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    assert got.UserCount == want.UserCount and got.ItemCount == want.ItemCount
    assert np.array_equal(got.innerUsers, want.innerUsers) and np.array_equal(got.innerItems, want.innerItems)
    assert _bits(got.GlobalMean) == _bits(want.GlobalMean)
    assert got._uraw is None                     # every id still has a row: the maps come from the rows as before


def test_change_after_remove(ml100k):
    rs = _rs()
    ts, u, i, r = _train(ml100k, True)
    removed = ts.Remove(u[:10], i[:10])
    got = removed.Change(rs.NewRawSet(u[10:20], i[10:20], np.full(10, 2.25)))
    want = r[10:].copy()
    want[:10] = 2.25
    assert np.array_equal(got.Ratings, want)
    assert np.array_equal(got.innerUsers, ts.innerUsers[10:])
    assert got.ConvertUserID(u[0]) == ts.ConvertUserID(u[0])
    assert _bits(got.GlobalMean) == _bits(rs.core._global_mean(want))


def test_refusals(ml100k):
    rs = _rs()
    ts, u, i, r = _train(ml100k)
    unrated = np.setdiff1d(np.unique(i), i[u == u[0]])[0]
    cases = [
        (RS_ERR_INVALID, lambda: ts.Remove([10 ** 6], [i[0]])),                 # unknown user
        (RS_ERR_INVALID, lambda: ts.Remove([u[0]], [10 ** 6])),                 # unknown item
        (RS_ERR_INVALID, lambda: ts.Remove([u[0]], [unrated])),                # a pair the set does not hold
        (RS_ERR_DUPLICATE, lambda: ts.Remove([u[0], u[0]], [i[0], i[0]])),
        (RS_ERR_INVALID, lambda: ts.Remove(u, i)),                              # nothing would be left
        (RS_ERR_INVALID, lambda: ts.Change(rs.NewRawSet([10 ** 6], [i[0]], [3.0]))),
        (RS_ERR_DUPLICATE, lambda: ts.Change(rs.NewRawSet([u[0], u[0]], [i[0], i[0]], [3.0, 2.0]))),
    ]
    for code, call in cases:
        with pytest.raises(rs.core.RsError) as e:
            call()
        assert e.value.code == code
    assert np.array_equal(ts.Users, u) and np.array_equal(ts.Ratings, r)
