"""The C++ mirror's KNN::RecommendGiven (host/core.hpp, host/recommend.cc --given) against KNN.RecommendGiven in
Python on ML-100K u1: the held-out u1.test ratings plus a new user and an unknown item, same users, raw item ids and
score bits."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import split

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("sim,knn_type,user_based", [("pearson", "centered", False), ("msd", "basic", True)])
def test_cpp_recommend_given_equals_python(ml100k, tmp_path, sim, knn_type, user_based):
    import recommend_sys_b200 as rs

    exe = Path(rs.core.__file__).resolve().parent / "rs_recommend"
    assert exe.exists(), "run __graft_entry__.build() (host/Makefile builds rs_recommend)"
    base, test = ml100k["u1_base"], ml100k["u1_test"]
    given = np.concatenate([test[:3000, :3], [[5000, 1, 4], [5000, 99999, 5], [5000, 50, 2]]])   # a new user
    data, gfile = tmp_path / "u1.base", tmp_path / "given"
    np.savetxt(data, base[:, :3], fmt="%d", delimiter="\t")
    np.savetxt(gfile, given, fmt="%d", delimiter="\t")
    n = 20
    out = subprocess.run([str(exe), str(data), sim, knn_type, str(int(user_based)), "40", str(n), "--given",
                          str(gfile)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = [x for x in out.stdout.split("\n") if x]
    got_users = [int(line.split()[0]) for line in lines]
    got_items = np.array([[int(v) for v in line.split()[1::2]] for line in lines], dtype=np.int64)
    got_bits = np.array([[int(v, 16) for v in line.split()[2::2]] for line in lines], dtype=np.uint64)
    sims = {"msd": rs.MSD, "pearson": rs.Pearson}
    ctors = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean}
    u, i, r = split(base)
    est = ctors[knn_type](rs.Parameters({"sim": sims[sim], "userBased": user_based, "k": 40}))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    gu, gi, gr = split(given)
    users, items, scores = est.RecommendGiven(rs.NewRawSet(gu, gi, gr), n)
    assert got_users == users.tolist() and users[-1] == 5000
    assert np.array_equal(got_items, items)
    assert np.array_equal(got_bits, scores.view(np.uint64))
    est.Close()
