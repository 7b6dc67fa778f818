"""Seeded ratings whose walk labels are far from the row ids (tests/test_walk_labels*.py).

Row r of the left dimension gets longer as r grows, in groups of 12 equal lengths (ties go by id), every seventh row
takes one of three shared lengths instead, and the last five rows are rated by most right ids: with RS_KNN_HEAVY_MIN =
POP_MIN they are the popular columns.  The ratings are listed row by row, so row r's first-appearance inner id is r
and the longest-first order runs against the ids."""
import numpy as np

N_LEFT, N_RIGHT, N_POP, POP_MIN = 300, 360, 5, 200


def left_lengths():
    r = np.arange(N_LEFT)
    n = 4 + 2 * (r // 12)
    n[r % 7 == 3] = np.array([10, 24, 40])[(r[r % 7 == 3] // 7) % 3]
    n[-N_POP:] = np.array([330, 300, 300, 280, 250])
    return n


def ratings(seed=5):
    """(left ids, right ids, integer ratings 1..5), listed by ascending left id"""
    rng = np.random.RandomState(seed)
    left, right = [], []
    for r, n in enumerate(left_lengths()):
        left.append(np.full(n, r))
        right.append(np.sort(rng.choice(N_RIGHT, n, replace=False)))
    left, right = np.concatenate(left), np.concatenate(right)
    return left, right, rng.randint(1, 6, len(left)).astype(np.float64)
