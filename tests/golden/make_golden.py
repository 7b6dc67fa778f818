"""Regenerates tests/golden/ml100k.npz from the reference's data fixture.

    python tests/golden/make_golden.py <reference checkout>/core/data/ml-100k

The MovieLens-100K fixture the reference's own tests run on (core/base_test.go:50-64 via core/data.go:270
LoadDataFromBuiltIn("ml-100k")) is stored here so that the tests need nothing outside the repository:
u.data (100,000 rows, md5 6e47046882bad158b0efbb84cd5cb987) and, for each row, which of the five fixed
folds u1..u5 that ship beside it in core/data/ml-100k/ holds it as a test row.  Each u{f}.test is the rows
of fold f and each u{f}.base the rows of the other folds, both sorted by (user, item), so the fold
column rebuilds all ten files exactly (tests/conftest.py load_ml100k; checked below before writing).
Parsing follows core/data.go:298-309: tab-separated, fields 0..2 through Atoi.
MovieLens data: GroupLens Research, University of Minnesota (see core/data/ml-100k/README).
"""
import hashlib
import sys
from pathlib import Path

import numpy as np

OUT = Path(__file__).resolve().parent
sys.path.insert(0, str(OUT.parent))


def load(src, name):
    rows = [ln.split("\t") for ln in (src / name).read_text().splitlines()]
    return np.array([[int(r[0]), int(r[1]), int(r[2])] for r in rows], dtype=np.int64)


def pack(u_data, tests):
    """u_data (n, 3) and the five test folds -> the stored columns {user, item, rating, fold}."""
    row = {(int(u), int(i)): x for x, (u, i, _) in enumerate(u_data)}
    assert len(row) == len(u_data), "duplicate (user, item) pairs"
    fold = np.zeros(len(u_data), dtype=np.uint8)
    for f, t in enumerate(tests, 1):
        fold[[row[(int(u), int(i))] for u, i, _ in t]] = f
    assert (fold > 0).all(), "a row of u.data is in no test fold"
    # max id 1682, ratings 1..5: narrow separate columns compress best
    return {"user": u_data[:, 0].astype(np.uint16), "item": u_data[:, 1].astype(np.uint16),
            "rating": u_data[:, 2].astype(np.uint8), "fold": fold}


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    src = Path(sys.argv[1])
    md5 = hashlib.md5((src / "u.data").read_bytes()).hexdigest()
    assert md5 == "6e47046882bad158b0efbb84cd5cb987", md5
    files = {"u_data": load(src, "u.data")}
    for f in range(1, 6):
        files[f"u{f}_base"] = load(src, f"u{f}.base")
        files[f"u{f}_test"] = load(src, f"u{f}.test")
    np.savez_compressed(OUT / "ml100k.npz", **pack(files["u_data"], [files[f"u{f}_test"] for f in range(1, 6)]))
    from conftest import load_ml100k

    back = load_ml100k()
    assert back.keys() == files.keys() and all(np.array_equal(back[k], files[k]) for k in files)
    print({k: v.shape for k, v in files.items()})
