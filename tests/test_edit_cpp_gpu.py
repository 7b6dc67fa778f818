"""The C++ mirror's KNN::Remove / KNN::Change (host/core.hpp, host/recommend.cc --remove / --change) against a Python
Fit of the edited TrainSet on ML-100K u1: every rating of one user and a seeded tenth of the rest removed, or a seeded
tenth changed; same lists, raw item ids and score bits."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import split

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("edit", ["remove", "change"])
@pytest.mark.parametrize("sim,knn_type,user_based", [("pearson", "zscore", False), ("msd", "centered", True)])
def test_cpp_edit_equals_refit(ml100k, tmp_path, sim, knn_type, user_based, edit):
    import recommend_sys_b200 as rs

    exe = Path(rs.core.__file__).resolve().parent / "rs_recommend"
    assert exe.exists(), "run __graft_entry__.build() (host/Makefile builds rs_recommend)"
    base = ml100k["u1_base"][:, :3]
    rows = np.sort(np.random.RandomState(61).choice(len(base), len(base) // 10, replace=False))
    if edit == "remove":
        rows = np.union1d(rows, np.flatnonzero(base[:, 0] == 2))     # user 2 loses every rating
    pairs = base[rows].copy()
    if edit == "change":
        pairs[:, 2] = 6 - pairs[:, 2]
    data, efile = tmp_path / "base", tmp_path / "edit"
    np.savetxt(data, base, fmt="%d", delimiter="\t")
    np.savetxt(efile, pairs, fmt="%d", delimiter="\t")
    users = [1, 2, 900, 943]
    n = 20
    out = subprocess.run([str(exe), str(data), sim, knn_type, str(int(user_based)), "40", str(n), f"--{edit}",
                          str(efile)] + [str(x) for x in users], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = [x for x in out.stdout.split("\n") if x]
    got_users = [int(line.split()[0]) for line in lines]
    got_items = np.array([[int(v) for v in line.split()[1::2]] for line in lines], dtype=np.int64)
    got_bits = np.array([[int(v, 16) for v in line.split()[2::2]] for line in lines], dtype=np.uint64)
    u, i, r = split(base)
    ts = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    pu, pi, pr = split(pairs)
    edited = ts.Remove(pu, pi) if edit == "remove" else ts.Change(rs.NewRawSet(pu, pi, pr))
    sims = {"msd": rs.MSD, "pearson": rs.Pearson}
    ctors = {"centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore}
    est = ctors[knn_type](rs.Parameters({"sim": sims[sim], "userBased": user_based, "k": 40}))
    est.Fit(edited)
    items, scores = est.Recommend(np.array(users), n)
    assert got_users == users
    assert np.array_equal(got_items, items)
    assert np.array_equal(got_bits, scores.view(np.uint64))
    est.Close()
