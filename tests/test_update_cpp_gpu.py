"""The C++ mirror's KNN::Update (host/core.hpp, host/recommend.cc --update) against a Fit of the union in Python on
ML-100K u1: the tail of u1.base and two new users added to a Fit of the rest, same lists, raw item ids and score bits."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import split

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("sim,knn_type,user_based", [("pearson", "zscore", False), ("msd", "centered", True)])
def test_cpp_update_equals_refit(ml100k, tmp_path, sim, knn_type, user_based):
    import recommend_sys_b200 as rs

    exe = Path(rs.core.__file__).resolve().parent / "rs_recommend"
    assert exe.exists(), "run __graft_entry__.build() (host/Makefile builds rs_recommend)"
    base = ml100k["u1_base"]
    m = len(base) - 6000
    add = np.concatenate([base[m:, :3], [[5000, 1, 4], [5000, 50, 2], [5001, 99999, 5], [3, 99999, 1]]])
    data, afile = tmp_path / "head", tmp_path / "tail"
    np.savetxt(data, base[:m, :3], fmt="%d", delimiter="\t")
    np.savetxt(afile, add, fmt="%d", delimiter="\t")
    users = [1, 2, 900, 943, 5000, 5001]
    n = 20
    out = subprocess.run([str(exe), str(data), sim, knn_type, str(int(user_based)), "40", str(n), "--update",
                          str(afile)] + [str(x) for x in users], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = [x for x in out.stdout.split("\n") if x]
    got_users = [int(line.split()[0]) for line in lines]
    got_items = np.array([[int(v) for v in line.split()[1::2]] for line in lines], dtype=np.int64)
    got_bits = np.array([[int(v, 16) for v in line.split()[2::2]] for line in lines], dtype=np.uint64)
    sims = {"msd": rs.MSD, "pearson": rs.Pearson}
    ctors = {"centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore}
    u, i, r = split(np.concatenate([base[:m, :3], add]))
    est = ctors[knn_type](rs.Parameters({"sim": sims[sim], "userBased": user_based, "k": 40}))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    items, scores = est.Recommend(np.array(users), n)
    assert got_users == users
    assert np.array_equal(got_items, items)
    assert np.array_equal(got_bits, scores.view(np.uint64))
    est.Close()
