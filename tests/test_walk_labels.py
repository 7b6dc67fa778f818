"""The walk's label rule and tools/walk_lookups.py's counts on the label fixture (CPU only)."""
import sys
from pathlib import Path

import numpy as np

from walk_fixture import N_LEFT, N_POP, POP_MIN, left_lengths, ratings

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
import walk_lookups as wl  # noqa: E402


def test_label_rule_longest_first_ties_by_id():
    left, _, _ = ratings()
    deg = np.bincount(left, minlength=N_LEFT)
    assert np.array_equal(deg, left_lengths())
    n_pop, lays = wl.layouts(left, N_LEFT, POP_MIN, 512)
    assert n_pop == N_POP
    _, lab, walk, n_cols = lays[1]
    order = sorted(range(N_LEFT), key=lambda i: (-deg[i], i))      # stable descending length
    assert [int(x) for x in np.argsort(lab)] == order
    assert sorted(order[:N_POP]) == list(range(N_LEFT - N_POP, N_LEFT))   # the popular rows come first
    assert np.array_equal(walk, lab >= 0) and n_cols == N_LEFT - N_POP
    assert sorted(lab[walk].tolist()) == list(range(n_cols))
    # the fixture does what it is for: labels far from the ids, and many ties
    assert np.corrcoef(lab[walk], np.flatnonzero(walk))[0, 1] < -0.8
    assert len(deg) - len(np.unique(deg)) > 200
    # the popular list caps at pop_max, and fewer than two rows are no list
    assert wl.layouts(left, N_LEFT, POP_MIN, 3)[0] == 3
    assert wl.layouts(left, N_LEFT, 320, 512)[0] == 0


def brute(left, right, col, walk, n_cols, jc):
    rows = {}
    for i, c in zip(left.tolist(), right.tolist()):
        rows.setdefault(c, []).append(i)
    lower = upper = nonempty = triples = 0
    n_q = (n_cols + jc - 1) // jc
    for i, c in zip(left.tolist(), right.tolist()):
        if not walk[i]:
            continue
        x = int(col[i])
        upper += n_q - x // jc
        mates = [int(col[j]) for j in rows[c] if walk[j] and j != i]
        triples += sum(y < x for y in mates)
        for q in range(x // jc + 1):
            lower += 1
            nonempty += any(y < x and y // jc == q for y in mates)
    return lower, upper, nonempty, triples


def test_walk_lookups_counts_match_brute_force():
    left, right, _ = ratings()
    n_pop, lays = wl.layouts(left, N_LEFT, POP_MIN, 512)
    got = {}
    for jc in (32, 128):
        for name, col, walk, n_cols in lays:
            got[name, jc] = wl.count(left, right, col, walk, n_cols, jc)
            assert got[name, jc] == brute(left, right, col, walk, n_cols, jc), (name, jc)
    ids, labels = (name for name, *_ in lays)
    for jc in (32, 128):
        assert got[labels, jc][3] == got[ids, jc][3]              # the same triples ...
        assert got[labels, jc][0] < got[ids, jc][0]               # ... in fewer lookups
