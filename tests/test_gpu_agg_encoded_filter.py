"""count / min / max / sum / avg ... group by under predicates on sorted-int-codec (PFOR_INT) columns on the GPU
(imm3_query_agg_ext with IMM3_AGG_ENCODED_FILTER: the block pipeline's filter front - blocks_prune, the lane / quad /
mini-block filter kernels, the offset scan - feeds agg_blocks_kernel<NG, NA, S, BS = true>) against the oracle, which
evaluates encoded predicates itself, against the dense-id twin, against numpy at 40 M rows, and across segment-sharded
ranks over the device exchange and the host merge."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

import oracle_lib as O
from agg_sum_ref import java_double, query_agg_ext
from helpers import conj, make_table, oracle_preds
from immutable3_b200 import (Avg, Count, EQ, Engine, GT, Imm3Error, LT, Match, Max, Min, NoSelect, Project, ProjectAgg, Query, SegmentManager,
                             Select, Sum)
from immutable3_b200 import _lib as L

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
_OPS = {Count: O.AGG_COUNT, Min: O.AGG_MIN, Max: O.AGG_MAX}
ROUTES = set()   # block filter routes taken by the queries of this module (test_every_route_was_taken)


def _route_kinds(route):
    kinds = set()
    for part in route.split(";"):
        name = part.split("/")[0]
        if name in ("blocks_prune", "blocks_filter_lane", "blocks_filter_quad", "blocks_filter", "offset_scan"):
            kinds.add(name)
    if "blocks_prune" not in kinds:
        kinds.add("unpruned")
    return kinds


def expected(orc, table, sel, aggs, group_by):
    """Columns of the query from the oracle: its own query_agg for Count / Min / Max, agg_sum_ref with a Sum / Avg."""
    if any(isinstance(a, (Sum, Avg)) for a in aggs):
        exp = query_agg_ext(orc, table, sel, aggs, group_by)
        return [np.asarray(c) for c in exp] if len(exp) and len(exp[0]) else []
    exp = orc.query_agg(table, oracle_preds(sel), [(_OPS[type(a)], a.col) for a in aggs], list(group_by))
    return [np.asarray(c) for c in exp.columns] if exp.nrows else []


def check(orc, eng, table, sel, aggs, group_by, route=None, **kw):
    """The query through the encoded filter against the oracle (rows, order, types, names, printed rows); returns the route."""
    sum_avg = any(isinstance(a, (Sum, Avg)) for a in aggs)
    exp = expected(orc, table, sel, aggs, group_by)
    n = len(exp[0]) if exp else 0
    with eng.execute(Query(table, sel, ProjectAgg(aggs, group_by)), sum_avg=sum_avg, encoded_filter=True, **kw) as got:
        assert got.nrows == n, (table, sel, aggs, group_by, got.nrows, n, got.route)
        assert got.ncols == len(group_by) + len(aggs)
        names = [got.col_name(c) for c in range(got.ncols)]
        assert names == list(group_by) + [f"{a.col}_{type(a).__name__.lower()}" for a in aggs]
        for a, agg in enumerate(aggs):
            want = {Sum: L.COL_INT64, Avg: L.COL_DOUBLE, Count: L.COL_COUNT, Min: L.COL_DOUBLE, Max: L.COL_DOUBLE}[type(agg)]
            assert got.col_type(len(group_by) + a) == want
        for c in range(got.ncols if n else 0):
            g = got.column(c)
            assert g.tobytes() == exp[c].astype(g.dtype).tobytes(), (table, sel, aggs, group_by, c, got.route)
        for i in range(min(n, 8)):
            want = [str(int(exp[len(group_by) + a][i])) if isinstance(agg, (Count, Sum)) else java_double(float(exp[len(group_by) + a][i]))
                    for a, agg in enumerate(aggs)]
            assert got.format_row(i) == "Row(" + ",".join(want) + ")"
        r = got.route
        assert got.kernel_launches == (len(r.split(";")) if r else 0)          # ("": a range that can never hold, no kernel)
    if route is not None:
        assert route in r, (route, r)
    ROUTES.update(_route_kinds(r))
    return r


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg_enc_filter")
    rng = np.random.default_rng(15)
    n = 30_000
    extra = [("day:PFOR_INT", (np.arange(n) // 1500).astype(np.int32)),                       # sorted, 20 values
             ("seq:PFOR_INT", (np.arange(n) + 7).astype(np.int32)),                           # strictly sorted
             ("e3:PFOR_INT", np.cumsum(rng.integers(0, 5000, n)).astype(np.int32))]           # sorted, irregular widths
    make_table(d, "p", n, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps", extra_cols=extra)          # quad kernel
    make_table(d, "pl", 60_000, 1024, 14, seed=4, id_codec="PFOR_INT", id_mode="sorted")                    # compresses: lane kernel
    make_table(d, "pr", 20_000, 128, 10, seed=3, id_codec="PFOR_INT", id_mode="random")      # raw mini-blocks, INT_MIN / INT_MAX
    make_table(d, "rag", 12_001, 100, 3, seed=2, id_codec="PFOR_INT", id_mode="steps")       # 41 segments, a 1-row tail block
    make_table(d, "one", 1, 8, 2, seed=2, id_codec="PFOR_INT")
    make_table(d, "tp", 50_000, 1024, 7, seed=6, id_codec="PFOR_INT", id_mode="steps")        # twins: same rows, encoded / dense id
    make_table(d, "td", 50_000, 1024, 7, seed=6, id_codec="DENSE_INT", id_mode="steps")
    orc, sm = O.Oracle(d), SegmentManager(d)
    yield d, orc, sm
    sm.close()
    orc.close()


def _ids(orc, table):
    return np.asarray(orc.query(table, [], ["id"]).columns[0]).astype(np.int64)


def window(lo, hi):
    return conj(Select("id", GT(int(lo))), Select("id", LT(int(hi))))


def _windows(ids, block):
    """Windows on the id column: inside one block, on block and mini-block edges, before / after the table, empty, EQ on
    the extremes, GT alone, LT alone."""
    n, lo, hi = len(ids), int(ids.min()), int(ids.max())
    at = lambda i: int(ids[min(max(i, 0), n - 1)])
    sels = [window(at(block + 5), at(block + block // 2)),                     # inside one block (sorted columns)
            window(at(block - 1), at(2 * block)),                              # on block edges
            window(at(block) - 1, at(3 * block) + 1),
            window(at(31), at(32 * 5)),                                        # on mini-block edges
            window(at(32) - 1, at(64)),
            window(lo - 100, lo + 1),                                          # before the table's first rows
            window(hi - 1, hi + 100),                                          # after its last rows
            window(lo - 1000, lo - 10),                                        # entirely before
            window(at(n // 2), at(n // 2) + 1),                                # empty: no integer strictly between
            Select("id", EQ(lo)), Select("id", EQ(hi)),
            Select("id", GT(at(n // 3))), Select("id", LT(at(n // 3))),
            window(lo - 1, hi + 1)]                                            # every row
    return sels


def test_windows_match_the_oracle(world):
    d, orc, sm = world
    eng = Engine(sm)
    shapes = [([Count("id"), Min("age"), Max("age")], ["state"]),
              ([Min("id"), Max("id")], []),                                    # the filtered column aggregated
              ([Count("age"), Max("id")], ["id"]),                             # ... and grouped
              ([Max("age"), Min("id"), Count("state")], ["state", "age"])]
    first = True
    for table, block in (("pl", 1024), ("p", 1024), ("pr", 128), ("rag", 100)):
        for sel in _windows(_ids(orc, table), block):
            for aggs, gb in shapes:
                r = check(orc, eng, table, sel, aggs, gb)
                assert r == "" or (r.startswith("agg_init;") and r.endswith("/bsel;agg_compact")), r
                if first:
                    assert "blocks_prune;blocks_filter_lane/" in r, r                 # pl's id compresses: pruned lane kernel
                    first = False
    for sel in (Select("id", GT(-10)), Select("id", LT(-10)), Select("id", EQ(int(_ids(orc, "one")[0])))):
        check(orc, eng, "one", sel, [Min("id"), Max("id"), Count("age")], ["id"])
        check(orc, eng, "one", sel, [Count("age")], [])


def test_mixed_and_two_encoded_predicates(world):
    d, orc, sm = world
    eng = Engine(sm)
    ids = _ids(orc, "p")
    w = window(ids[3000], ids[20000])
    first = True
    for sel in (conj(w, Select("age", GT(18))),                                        # mini-block kernel, unpruned
                conj(w, Select("state", Match(["CA", "NY"]))),
                conj(Select("id", GT(int(ids[5000]))), Select("seq", LT(25_000))),     # two encoded columns: pruned, mini
                conj(w, Select("day", EQ(7))),
                conj(w, Select("e3", GT(1_000_000)), Select("age", LT(50)))):
        for aggs, gb in (([Count("id"), Min("age"), Max("age")], ["state"]), ([Min("seq"), Max("e3")], ["day"]), ([Count("age")], ["seq"])):
            r = check(orc, eng, "p", sel, aggs, gb)
            if first:
                assert ";blocks_filter/s=" in r and "blocks_prune" not in r, r
                first = False


def test_block_filter_routes(world, monkeypatch):
    d, orc, sm = world
    eng = Engine(sm)
    ids = _ids(orc, "pl")
    sels = [window(ids[1500], ids[9000]), window(ids[0] - 5, ids[-1] + 5), Select("id", GT(int(ids[58000])))]
    aggs, gb = [Count("id"), Min("age"), Max("age")], ["state"]
    for env, want, gone in ((("IMM3_NO_LANE", "1"), ";blocks_filter_quad/", None),
                            (("IMM3_NO_QUAD", "1"), ";blocks_filter/s=", None),
                            (("IMM3_NO_PRUNE", "1"), "agg_init;blocks_filter_lane/", "blocks_prune"),
                            (("IMM3_LANE_WARPS", "4"), "/w=4/", None),
                            (("IMM3_PATH", "fused"), "blocks_prune;blocks_filter_lane/", None),      # Project switches do not apply
                            (("IMM3_NO_HYBRID", "1"), "blocks_prune;blocks_filter_lane/", None)):
        monkeypatch.setenv(*env)
        for i, sel in enumerate(sels):
            r = check(orc, eng, "pl", sel, aggs, gb)
            if i == 0:
                assert want in r and (gone is None or gone not in r), (env, r)
                if env[0] == "IMM3_LANE_WARPS":
                    assert ";offset_scan;agg_blocks<" in r, r                 # a lane kernel of 4 warps does not scan inline
        monkeypatch.delenv(env[0])
    with SegmentManager(d, flags=L.OPEN_NO_STATS) as nostats:                  # no block statistics: nothing to prune from
        e2 = Engine(nostats)
        for i, sel in enumerate(sels):
            r = check(orc, e2, "pl", sel, aggs, gb)
            if i == 0:
                assert r.startswith("agg_init;blocks_filter_lane/"), r


def test_every_instantiation(world):
    """agg_blocks_kernel<NG, NA, S, true>: NG in {0, 1, 2, 4} x NA in {1 .. 4, 8} without a Sum, NA in {2, 3, 4, 8} with one."""
    d, orc, sm = world
    eng = Engine(sm)
    ids = _ids(orc, "p")
    sel = window(ids[700], ids[26000])
    many = [Min("id"), Count("id"), Max("seq"), Min("age"), Max("age"), Count("state"), Max("id"), Min("day")]
    by_na = {2: [Sum("age")], 3: [Sum("id"), Avg("age")], 4: [Avg("age"), Min("id"), Max("age")],
             8: [Sum("age"), Sum("id"), Avg("age"), Min("age"), Max("id"), Avg("id"), Min("id")]}
    for gb, ng in (([], 0), (["state"], 1), (["state", "age"], 2), (["day", "state", "age"], 4)):
        for na in (1, 2, 3, 4, 5, 8):
            check(orc, eng, "p", sel, many[:na], gb, route=f";agg_blocks<{ng},{8 if na > 4 else na}>/bsel;agg_compact")
        for na, aggs in by_na.items():
            check(orc, eng, "p", sel, aggs, gb, route=f";agg_blocks<{ng},{na}>/sum/bsel;agg_compact")
    for aggs in ([Sum("id"), Avg("id"), Count("id")], [Sum("age"), Avg("seq")]):              # Sum / Avg over other windows
        for s in _windows(ids, 1024)[:6]:
            check(orc, eng, "p", s, aggs, ["state"])


def test_twins_agree(world):
    """The encoded table through the block filter gives the columns the dense-id twin gives on its row-space path."""
    d, orc, sm = world
    eng = Engine(sm)
    ids = _ids(orc, "td")
    for sel in _windows(ids, 1024) + [conj(window(ids[4000], ids[40000]), Select("age", GT(18)))]:
        for aggs, gb in (([Count("id"), Min("age"), Max("age")], ["state"]), ([Min("id"), Max("id")], ["age"]),
                         ([Sum("age"), Avg("id"), Count("id")], ["state"])):
            sa = any(isinstance(a, (Sum, Avg)) for a in aggs)
            q = lambda t: Query(t, sel, ProjectAgg(aggs, gb))
            with eng.execute(q("tp"), sum_avg=sa, encoded_filter=True) as a, eng.execute(q("td"), sum_avg=sa) as b:
                assert ("/bsel" in a.route) == (a.route != "") and "/bsel" not in b.route   # ("": a range that never holds)
                assert a.nrows == b.nrows and a.ncols == b.ncols
                for c in range(a.ncols):
                    assert a.col_name(c) == b.col_name(c) and a.col_type(c) == b.col_type(c)
                    assert a.column(c).tobytes() == b.column(c).tobytes(), (sel, aggs, gb, c)


def test_flag_changes_nothing_without_an_encoded_predicate(world):
    d, orc, sm = world
    eng = Engine(sm)
    for table in ("p", "td", "rag"):
        for sel in (NoSelect, Select("age", GT(18)), conj(Select("state", Match(["CA"])), Select("age", LT(40)))):
            for aggs, gb in (([Count("id"), Min("id"), Max("age")], ["state"]), ([Count("age")], ["id"]), ([Sum("age"), Avg("id")], ["state"])):
                sa = any(isinstance(x, (Sum, Avg)) for x in aggs)
                q = Query(table, sel, ProjectAgg(aggs, gb))
                with eng.execute(q, sum_avg=sa) as a, eng.execute(q, sum_avg=sa, encoded_filter=True) as b:
                    assert a.route == b.route and "/bsel" not in b.route
                    assert a.nrows == b.nrows and a.kernel_launches == b.kernel_launches
                    for c in range(a.ncols):
                        assert a.col_name(c) == b.col_name(c) and a.col_type(c) == b.col_type(c)
                        assert a.column(c).tobytes() == b.column(c).tobytes()
                    for i in range(min(a.nrows, 5)):
                        assert a.format_row(i) == b.format_row(i)


@pytest.mark.parametrize("table", ["p", "pl"])
@pytest.mark.parametrize("prune", [True, False])
def test_stale_bitmap_words_are_never_read(world, monkeypatch, prune, table):
    """A window whose edges cut blocks X and Y writes their words; Project queries (C4: a window on id, id projected) write
    other blocks' words; then windows that select X and Y wholly or not at all must not see any of those words."""
    d, orc, sm = world
    eng = Engine(sm)
    if not prune:
        monkeypatch.setenv("IMM3_NO_PRUNE", "1")
    ids = _ids(orc, table)                                                      # canonical order: blocks of 1024 rows
    X, Y = 5, 17
    blk = lambda b: ids[b * 1024:(b + 1) * 1024]
    mid = lambda b: int(ids[b * 1024 + 500])
    aggs, gb = [Count("id"), Min("age"), Max("age"), Min("id")], ["state"]
    selected = lambda lo, hi, b: int(((blk(b) > lo) & (blk(b) < hi)).sum())   # rows of block b in the window (lo, hi)
    cut_b = (mid(X), mid(Y))                                                    # edges inside X and inside Y
    for b in (X, Y):
        assert 0 < selected(*cut_b, b) < 1024
    whole_b = [(int(blk(X).min()) - 1, int(blk(Y).max()) + 1),                  # X and Y wholly selected
               (int(blk(X).max()), int(blk(Y).min())),                          # X and Y not at all
               (int(blk(X).min()) - 1, int(blk(Y).min()))]                      # X wholly, Y not at all
    assert [(selected(*w, X), selected(*w, Y)) for w in whole_b] == [(1024, 1024), (0, 0), (1024, 0)]
    cut, wholly = window(*cut_b), [window(*w) for w in whole_b]
    for rnd in range(3):
        check(orc, eng, table, cut, aggs, gb)
        for k in range(3):
            lo, hi = mid(2 + 7 * k + rnd), mid(9 + 7 * k + rnd)
            exp = orc.query(table, oracle_preds(window(lo, hi)), ["id"], limit=0)
            with eng.execute(Query(table, window(lo, hi), Project(["id"]))) as r:
                assert r.nrows == exp.nrows and np.array_equal(r.column(0), exp.columns[0])
        for sel in wholly:
            check(orc, eng, table, sel, aggs, gb)
            check(orc, eng, table, sel, [Sum("age"), Avg("id")], ["state"])


def test_cold_path_and_overflow(world, monkeypatch):
    d, orc, sm = world
    eng = Engine(sm)
    ids = _ids(orc, "p")
    sel = window(ids[100], ids[29000])
    assert len(expected(orc, "p", sel, [Count("age")], ["seq"])[0]) > 20_000
    check(orc, eng, "p", sel, [Count("age"), Min("id")], ["seq"])               # > 256 groups per CTA: the global table
    check(orc, eng, "p", sel, [Sum("age"), Avg("id")], ["seq"])
    monkeypatch.setenv("IMM3_AGG_SLOTS", "64")
    for aggs in ([Min("id")], [Sum("age")]):
        with pytest.raises(Imm3Error) as e:
            eng.execute(Query("p", sel, ProjectAgg(aggs, ["seq"])), sum_avg=True, encoded_filter=True)
        assert e.value.status == L.ERR_UNSUPPORTED and "groups" in e.value.message   # reported, not truncated
    monkeypatch.delenv("IMM3_AGG_SLOTS")
    check(orc, eng, "p", sel, [Min("id"), Max("id")], ["state"])                 # the handle is fine afterwards


def test_every_route_was_taken():
    if not ROUTES:
        pytest.skip("no query of this module ran before this test")
    assert {"blocks_prune", "unpruned", "blocks_filter_lane", "blocks_filter_quad", "blocks_filter", "offset_scan"} <= ROUTES, ROUTES


# ---- 40 M rows against numpy ----------------------------------------------------------------------------------------------

def _numpy_group(keys, mask, vals):
    k, v = keys[mask], vals[mask]
    uniq, first, inv = np.unique(k, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    g = rank[inv.reshape(-1)]
    cnt = np.bincount(g, minlength=len(uniq))
    mn = np.full(len(uniq), np.iinfo(np.int64).max)
    mx = np.full(len(uniq), np.iinfo(np.int64).min)
    np.minimum.at(mn, g, v.astype(np.int64))
    np.maximum.at(mx, g, v.astype(np.int64))
    return uniq[order], cnt, mn, mx


def test_40m_rows_against_numpy(tmp_path, monkeypatch):
    from immutable3_b200.loader import synth_write

    n = 40_000_000
    synth_write(str(tmp_path), "t", n, 1024, 1000, L.CODEC_PFOR_INT)
    with O.Oracle(tmp_path) as orc:
        raw = orc.query("t", [], ["id", "state", "age"])                 # the segment files, decoded in canonical order
    ids, states, ages = (np.asarray(c) for c in raw.columns)
    assert len(ids) == n
    srt = np.sort(ids.astype(np.int64))
    with SegmentManager(tmp_path) as sm:
        eng = Engine(sm)
        for frac in (0.01, 0.5, 1.0):
            lo = int(srt[int(n * (0.5 - frac / 2))]) - 1 if frac < 1 else int(srt[0]) - 1
            hi = int(srt[min(n - 1, int(n * (0.5 + frac / 2)))]) if frac < 1 else int(srt[-1]) + 1
            sel = window(lo, hi)
            inwin = (ids.astype(np.int64) > lo) & (ids.astype(np.int64) < hi)
            for mixed in (False, True):
                s = conj(sel, Select("age", GT(18))) if mixed else sel
                m = inwin & (ages > 18) if mixed else inwin
                keys, cnt, mn, mx = _numpy_group(states, m, ages)
                for prune in ((True, False) if not mixed else (True,)):
                    if not prune:
                        monkeypatch.setenv("IMM3_NO_PRUNE", "1")
                    q = Query("t", s, ProjectAgg([Count("id"), Min("age"), Max("age"), Sum("age")], ["state"]))
                    with eng.execute(q, sum_avg=True, encoded_filter=True) as r:
                        assert ("blocks_prune" in r.route) == (prune and not mixed), r.route
                        assert np.array_equal(r.column(0), keys) and np.array_equal(r.column(1), cnt), (frac, mixed, prune)
                        assert np.array_equal(r.column(2), mn.astype(np.float64)) and np.array_equal(r.column(3), mx.astype(np.float64))
                        s_ = np.zeros(len(cnt), np.int64)
                        _, first, inv = np.unique(states[m], return_index=True, return_inverse=True)
                        order = np.argsort(first, kind="stable")
                        rank = np.empty_like(order)
                        rank[order] = np.arange(len(order))
                        np.add.at(s_, rank[inv.reshape(-1)], ages[m].astype(np.int64))
                        assert r.column(4).tolist() == s_.tolist()
                    monkeypatch.delenv("IMM3_NO_PRUNE", raising=False)


# ---- across ranks ---------------------------------------------------------------------------------------------------------

def _cases(ids):
    w = lambda a, b: window(ids[int(a * (len(ids) - 1))], ids[int(b * (len(ids) - 1))])   # (a, b: fractions of the rows)
    return [(w(0.1, 0.7), [Count("id"), Min("age"), Max("age")], ["state"]),
            (w(0.0, 1.0), [Min("id"), Max("id")], []),
            (window(ids[0] - 10, ids[0] - 1), [Count("age")], ["state"]),                  # nothing matches anywhere
            (conj(w(0.03, 0.8), Select("age", GT(18))), [Count("id"), Max("id")], ["state"]),
            (w(0.02, 0.3), [Sum("age"), Avg("id")], ["state"]),
            (w(0.07, 0.9), [Count("age"), Min("id")], ["id"])]


def _worker(rank, world, data_dir, port, out_dir, mode):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch
    import torch.distributed as dist

    import oracle_lib as O
    from immutable3_b200 import Engine, ProjectAgg, Query, SegmentManager
    from immutable3_b200.dist import CudaExecutor, ShardedEngine

    ndev = torch.cuda.device_count()
    dev = rank % ndev
    backend = "nccl" if (mode == "device" and ndev >= world) else "gloo"
    if backend == "nccl":
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    os.environ["IMM3_COMM_TIMEOUT_MS"] = "10000"
    try:
        with SegmentManager(data_dir, device=dev, rank=rank, world=world) as sm, O.Oracle(data_dir) as whole:
            if mode == "device":
                sm.comm_connect()
            eng = Engine(sm)
            sh = ShardedEngine(CudaExecutor(eng), collective_device="cuda" if backend == "nccl" else "cpu")
            for sel, aggs, gb in _cases(_ids(whole, "p")):
                sa = any(isinstance(a, (Sum, Avg)) for a in aggs)
                q = Query("p", sel, ProjectAgg(aggs, gb))
                exp = expected(whole, "p", sel, aggs, gb)
                n = len(exp[0]) if exp else 0
                res = sh.execute_agg(q, sum_avg=sa, encoded_filter=True)
                assert res.total == n and len(res.columns) == len(gb) + len(aggs), (mode, rank, aggs, gb, res.total, n)
                for c in range(len(res.columns) if n else 0):
                    assert res.columns[c].tobytes() == exp[c].astype(res.columns[c].dtype).tobytes(), (mode, rank, aggs, gb, c)
                if mode == "device":
                    with eng.execute_agg_global(q, sum_avg=sa, encoded_filter=True) as r:
                        assert r.global_count == n
                        assert r.route.endswith("agg_exchange;agg_init;agg_merge;agg_compact"), r.route
                        assert "/bsel;agg_compact;agg_exchange" in r.route or r.route.startswith("agg_exchange"), r.route
                        assert r.kernel_launches == len(r.route.split(";")), (r.kernel_launches, r.route)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def _tables(tmp_path, small=False):
    data = tmp_path / "data"
    if small:   # one segment: ranks past the first own an empty slice
        make_table(data, "p", 2000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    else:
        make_table(data, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    return data


@pytest.mark.parametrize("world, mode", [(2, "device"), (3, "device"), (2, "host"), (3, "host")])
def test_sharded(tmp_path, world, mode):
    data = _tables(tmp_path)
    port = 45700 + (os.getpid() % 2000) + world + (10 if mode == "host" else 0)
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path), mode), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


@pytest.mark.parametrize("mode", ["device", "host"])
def test_sharded_four_ranks_with_empty_slices(tmp_path, mode):
    data = _tables(tmp_path, small=True)
    port = 48700 + (os.getpid() % 1000) + (10 if mode == "host" else 0)
    mp.spawn(_worker, args=(4, str(data), port, str(tmp_path), mode), nprocs=4, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(4))
