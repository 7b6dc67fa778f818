import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _built():
    """Everything is built in-tree by __graft_entry__.build(); make sure it happened."""
    import __graft_entry__ as g

    pkg = ROOT / "recommend-sys_b200"
    if not ((pkg / "librs_knn_b200.so").exists() and (pkg / "librs_host.so").exists()
            and (ROOT / "oracle" / "libknn_oracle.so").exists()):
        g.build()


def load_ml100k():
    """The reference's data fixture (core/data/ml-100k), see tests/golden/make_golden.py: "u_data" and the
    fixed folds "u1_base" .. "u5_test" as int64 (n, 3) arrays of (user, item, rating).  A fold's files are
    the rows of u.data sorted by (user, item): u{f}_test those stored with fold f, u{f}_base the others."""
    g = np.load(ROOT / "tests" / "golden" / "ml100k.npz")
    u_data, fold = np.stack([g["user"], g["item"], g["rating"]], axis=1).astype(np.int64), g["fold"]
    order = np.lexsort((u_data[:, 1], u_data[:, 0]))
    out = {"u_data": u_data}
    for f in range(1, 6):
        test = fold[order] == f
        out[f"u{f}_base"] = u_data[order[~test]]
        out[f"u{f}_test"] = u_data[order[test]]
    return out


@pytest.fixture(scope="session")
def ml100k():
    return load_ml100k()


def split(a):
    return a[:, 0], a[:, 1], a[:, 2].astype(np.float64)


def bits_equal(a, b):
    """Bit-exact equality of float64 arrays where any NaN equals any NaN."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False
    return np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))
