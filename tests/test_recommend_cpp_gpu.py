"""The C++ mirror's KNN::Recommend (host/core.hpp, driven by host/recommend.cc) against KNN.Recommend in Python on
ML-100K: the same raw item ids and the same score bits, with k changed after Fit."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import split

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("sim,knn_type,user_based,k", [("pearson", "centered", False, 30), ("msd", "basic", True, 50),
                                                       ("cosine", "zscore", False, 40)])
def test_cpp_recommend_equals_python(ml100k, tmp_path, sim, knn_type, user_based, k):
    import recommend_sys_b200 as rs

    exe = Path(rs.core.__file__).resolve().parent / "rs_recommend"
    assert exe.exists(), "run __graft_entry__.build() (host/Makefile builds rs_recommend)"
    base = ml100k["u1_base"]
    data = tmp_path / "u1.base"
    np.savetxt(data, base[:, :3], fmt="%d", delimiter="\t")
    users = [1, 5, 943, 10 ** 9, 1, 200]                       # an unknown user (newID) and a duplicate
    n = 25
    out = subprocess.run([str(exe), str(data), sim, knn_type, str(int(user_based)), str(k), str(n)]
                         + [str(x) for x in users], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.split("\n")[:len(users)]
    got_items = np.array([[int(v) for v in line.split()[1::2]] for line in lines], dtype=np.int64)
    got_bits = np.array([[int(v, 16) for v in line.split()[2::2]] for line in lines], dtype=np.uint64)
    assert [int(line.split()[0]) for line in lines] == users

    sims = {"cosine": rs.Cosine, "msd": rs.MSD, "pearson": rs.Pearson}
    ctors = {"basic": rs.NewKNN, "centered": rs.NewKNNWithMean, "zscore": rs.NewKNNWithZScore}
    u, i, r = split(base)
    est = ctors[knn_type](rs.Parameters({"sim": sims[sim], "userBased": user_based, "k": 40}))
    est.Fit(rs.NewTrainSet(rs.NewRawSet(u, i, r)))
    est.SetParams(rs.Parameters({"sim": sims[sim], "userBased": user_based, "k": k}))
    items, scores = est.Recommend(np.array(users), n)
    assert np.array_equal(got_items, items)
    assert np.array_equal(got_bits, scores.view(np.uint64))
    raw = np.empty(est.Data.ItemCount, np.int64)                  # inner -> raw item id
    raw[est.Data.innerItems] = est.Data.Items
    assert np.array_equal(items[3], raw[:n]) and (scores[3] == est.GlobalMean).all()   # newID: the first n items
    assert np.array_equal(items[0], items[4])
    est.Close()
