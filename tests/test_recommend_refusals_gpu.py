"""The exact return code of every refusal of the ten recommendation entry points (rs_knn_score_all[_device],
rs_knn_recommend[_device], rs_knn_*_sharded_device, rs_knn_*_given[_device]), called through the C ABI so that null
pointers, bad sides and out-of-range counts reach the library unchanged.  The families differ on purpose: a top-k-only
handle is RS_ERR_INVALID for the by-id and sharded entry points but RS_ERR_UNSUPPORTED for the given ones, by-id entry
points return before their null check when n == 0, and only the host by-id variants refuse query ids outside [-1, n)."""
import ctypes as C

import numpy as np
import pytest

from conftest import split
import test_recommend_gpu as rg

pytestmark = pytest.mark.gpu

OK, INVALID, UNSUPPORTED, DUPLICATE = 0, -1, -3, -5
LEFT, RIGHT = 0, 1
NQ = 4                       # queries the buffers hold

# entry point -> (family, lists, host): family "id" / "sharded" / "given", lists: the top-n_top form
ENTRIES = {
    "score_all": ("id", False, True),
    "score_all_device": ("id", False, False),
    "recommend": ("id", True, True),
    "recommend_device": ("id", True, False),
    "score_all_sharded_device": ("sharded", False, False),
    "recommend_sharded_device": ("sharded", True, False),
    "score_all_given": ("given", False, True),
    "score_all_given_device": ("given", False, False),
    "recommend_given": ("given", True, True),
    "recommend_given_device": ("given", True, False),
}
BY_ID = [e for e, (f, _, _) in ENTRIES.items() if f == "id"]
SHARDED = [e for e, (f, _, _) in ENTRIES.items() if f == "sharded"]
GIVEN = [e for e, (f, _, _) in ENTRIES.items() if f == "given"]
LISTS = [e for e, (_, t, _) in ENTRIES.items() if t]


class Buffers:
    """Host and device arrays for NQ queries: ids, one-entry lists, score rows and lists of up to 512."""

    def __init__(self, width):
        import torch

        self.host = {"q": np.zeros(NQ, np.int32), "ptr": np.arange(NQ + 1, dtype=np.int64),
                     "ids": np.full(NQ, 3, np.int32), "vals": np.ones(NQ), "out": np.empty(NQ * width),
                     "ti": np.empty(NQ * 512, np.int32), "ts": np.empty(NQ * 512)}
        self.dev = {k: torch.from_numpy(v).cuda() for k, v in self.host.items()}
        torch.cuda.synchronize()

    def ptr(self, host, name):
        return self.host[name].ctypes.data if host else self.dev[name].data_ptr()

    def set(self, host, name, values):
        import torch

        a = np.asarray(values, dtype=self.host[name].dtype)
        if host:
            self.host[name][:len(a)] = a
        else:
            self.dev[name][:len(a)] = torch.from_numpy(a).cuda()
            torch.cuda.synchronize()


def call(buf, entry, h, side=LEFT, n=1, n_top=5, null=()):
    """The return code of `entry` on handle h; pointer arguments named in `null` are passed as NULL."""
    import recommend_sys_b200 as rs

    family, lists, host = ENTRIES[entry]
    names = ("ptr", "ids", "vals") if family == "given" else ("q",)

    def p(name):
        return None if name in null else buf.ptr(host, name)

    args = [h, side] + [p(x) for x in names] + [n]
    args += [n_top, p("ti"), p("ts")] if lists else [p("out")]
    rc = getattr(rs.core.knn_lib(), "rs_knn_" + entry)(*args)
    if rc == OK:
        assert rs.core.knn_lib().rs_knn_synchronize(h) == OK
    return rc


def expect(buf, entries, h, want, **kw):
    got = {e: call(buf, e, h, **kw) for e in entries}
    assert got == {e: want for e in entries}, kw


def _shards(u, i, r, mirror):
    shards = [rg._fit(u, i, r, "msd", "basic", True, extra={"shardCount": 2, "shardIndex": s}) for s in range(2)]
    for s in shards:
        s._h.synchronize()
    if mirror:
        for s in shards:
            s._h.peer_import_local([x._h for x in shards])
            s._h.mirror()
    return shards


def test_refusal_codes(ml100k):
    import recommend_sys_b200 as rs

    u, i, r = split(ml100k["u1_base"])
    buf = Buffers(2000)
    every = list(ENTRIES)

    # not fitted
    fresh = rs.core._Handle()
    expect(buf, every, fresh.h, INVALID)
    fresh.close()

    # top-k-only handle: the given entry points check the store first
    e = rg._fit(u, i, r, "msd", "basic", True, extra={"store": "topk", "topk": 40, "simPath": "stream"})
    expect(buf, BY_ID + SHARDED, e._h.h, INVALID)
    expect(buf, GIVEN, e._h.h, UNSUPPORTED)
    expect(buf, BY_ID + SHARDED, e._h.h, INVALID, side=7)           # the store is checked before the side
    expect(buf, GIVEN, e._h.h, UNSUPPORTED, side=7)
    e.Close()

    # a full handle: everything that checks the arguments
    full = rg._fit(u, i, r, "msd", "basic", True, extra={"simPath": "stream"})
    h = full._h.h
    expect(buf, SHARDED, h, INVALID)                                # not a row shard
    for side in (-1, 2):
        expect(buf, BY_ID + GIVEN, h, INVALID, side=side)
    for n in (-1, 1 << 31):
        expect(buf, BY_ID + GIVEN, h, INVALID, n=n)
    for n_top in (0, 513):
        expect(buf, [x for x in BY_ID + GIVEN if x in LISTS], h, INVALID, n_top=n_top)
        expect(buf, [x for x in BY_ID + GIVEN if x in LISTS], h, INVALID, n=0, n_top=n_top)   # n_top before n == 0
    for entry in BY_ID + GIVEN:
        family, lists, _ = ENTRIES[entry]
        names = (("ptr", "ids", "vals") if family == "given" else ("q",)) + (("ti", "ts") if lists else ("out",))
        for name in names:
            assert call(buf, entry, h, null=(name,)) == INVALID, (entry, name)
        assert call(buf, entry, h, n=0, null=names) == OK, entry
    # query ids outside [-1, n_left): refused by the host variants, cold start on the device
    for bad in (-2, full._h.n_left):
        buf.set(True, "q", [bad])
        buf.set(False, "q", [bad])
        expect(buf, ["score_all", "recommend"], h, INVALID)
        expect(buf, ["score_all_device", "recommend_device"], h, OK)
    buf.set(True, "q", [0])
    buf.set(False, "q", [0])
    # the lists themselves, validated on the host (ptr[0]) or the device
    for host in (True, False):
        buf.set(host, "ptr", [-1])
    expect(buf, GIVEN, h, INVALID)
    for host in (True, False):
        buf.set(host, "ptr", [0, 2, 1])
    expect(buf, GIVEN, h, INVALID, n=2)                             # decreasing
    for host in (True, False):
        buf.set(host, "ptr", [0, 1, 3])
        buf.set(host, "ids", [3, 4, 4])
    expect(buf, GIVEN, h, DUPLICATE, n=2)
    for host in (True, False):
        buf.set(host, "ptr", np.arange(NQ + 1))
        buf.set(host, "ids", [full._h.n_right])
    expect(buf, GIVEN, h, INVALID)                                  # an id out of range
    for host in (True, False):
        buf.set(host, "ids", [3])
        buf.set(host, "vals", [np.nan])
    expect(buf, GIVEN, h, INVALID)                                  # a NaN rating
    for host in (True, False):
        buf.set(host, "vals", [1.0])
    expect(buf, GIVEN, h, UNSUPPORTED, n=(1 << 31) - 1)             # n_left + n beyond 2^31 - 1 (left lists)
    expect(buf, BY_ID + GIVEN, h, OK)
    expect(buf, BY_ID + GIVEN, h, OK, side=RIGHT)
    full._h.set_k(257, 1)
    expect(buf, BY_ID + GIVEN, h, UNSUPPORTED)
    expect(buf, BY_ID + GIVEN, h, UNSUPPORTED, n=0, n_top=0)        # k before n_top and n == 0
    full.Close()

    # left lists the model cannot score: no baseline bias, or not the exact Pearson matrix
    for sim, typ, extra in (("msd", "baseline", {}), ("pearson_baseline", "basic", {}),
                            ("pearson", "basic", {"pearsonMode": "sums"})):
        e = rg._fit(u, i, r, sim, typ, True, extra=extra)
        expect(buf, GIVEN, e._h.h, UNSUPPORTED)
        expect(buf, GIVEN, e._h.h, OK, side=RIGHT)
        expect(buf, GIVEN, e._h.h, UNSUPPORTED, null=("ptr",))      # before the null check
        e.Close()

    # cyclic shards before the mirror step, then after it
    shards = _shards(u, i, r, mirror=False)
    for s in shards:
        expect(buf, BY_ID + GIVEN, s._h.h, UNSUPPORTED)
        expect(buf, SHARDED, s._h.h, INVALID)
    for s in shards:
        s.Close()
    shards = _shards(u, i, r, mirror=True)
    s = shards[0]._h.h
    expect(buf, BY_ID + GIVEN, s, UNSUPPORTED)
    expect(buf, SHARDED, s, OK)
    expect(buf, SHARDED, s, OK, side=RIGHT)
    for side in (-1, 2):
        expect(buf, SHARDED, s, INVALID, side=side)
    for n in (-1, 1 << 31):
        expect(buf, SHARDED, s, INVALID, n=n)
    for n_top in (0, 513):
        expect(buf, ["recommend_sharded_device"], s, INVALID, n_top=n_top)
        expect(buf, ["recommend_sharded_device"], s, INVALID, n=0, n_top=n_top)
    for entry in SHARDED:
        names = ("q",) + (("ti", "ts") if ENTRIES[entry][1] else ("out",))
        for name in names:
            assert call(buf, entry, s, null=(name,)) == INVALID, (entry, name)
        assert call(buf, entry, s, n=0, null=names) == OK, entry
    buf.set(False, "q", [-2])
    expect(buf, SHARDED, s, OK)                                     # cold start, as the plain device variants
    buf.set(False, "q", [0])
    shards[0]._h.set_k(257, 1)
    expect(buf, SHARDED, s, UNSUPPORTED)
    for x in shards:
        x.Close()

    # contiguous row shard
    e = rg._fit(u, i, r, "msd", "basic", True, extra={"rowBegin": 0, "rowEnd": 100, "simPath": "stream"})
    expect(buf, BY_ID + GIVEN, e._h.h, UNSUPPORTED)
    expect(buf, SHARDED, e._h.h, OK)
    e.Close()

    # Slope One: a full handle is not a row shard, a contiguous shard of it is refused for the similarity
    train = rs.NewTrainSet(rs.NewRawSet(u, i, r))
    for params, sharded_rc in (({}, INVALID), ({"rowBegin": 0, "rowEnd": 100}, UNSUPPORTED)):
        so = rs.NewSlopeOne(rs.Parameters(params))
        so.Fit(train)
        expect(buf, BY_ID + GIVEN, so._h.h, UNSUPPORTED, side=RIGHT)
        expect(buf, SHARDED, so._h.h, sharded_rc, side=RIGHT)
        so.Close()
