"""Sum / Avg ... group by on the GPU (imm3_query_agg_ext; k_agg.cuh's SUM instantiations of agg_kernel and
agg_blocks_kernel) against a restatement over the oracle's rows (agg_sum_ref.py), against numpy at 40 M rows, and across
segment-sharded ranks (IMM3_AGG_GLOBAL over the device exchange, ShardedEngine.execute_agg over the host exchange).
A group of more than 2^32 rows, which imm3_query_agg_ext refuses, would need a 4.3 G-row table: that check is not tested here."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

import oracle_lib as O
from agg_sum_ref import java_double, query_agg_ext
from helpers import conj, make_table
from immutable3_b200 import (Avg, Count, EQ, Engine, GT, Imm3Error, LT, Match, Max, Min, NoSelect, ProjectAgg, Query, SegmentManager, Select,
                             Sum)
from immutable3_b200 import _lib as L

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
I32_MIN, I32_MAX = -2**31, 2**31 - 1


def check_ext(orc, eng, table, sel, aggs, group_by, route=None):
    exp = query_agg_ext(orc, table, sel, aggs, group_by)
    with eng.execute(Query(table, sel, ProjectAgg(aggs, group_by)), sum_avg=True) as got:
        assert got.ncols == len(group_by) + len(aggs)
        n = len(exp[0]) if len(exp) and len(exp[0]) else 0
        assert got.nrows == n, (table, sel, aggs, group_by, got.nrows, n)
        if route:
            assert route in got.route, (route, got.route)
        assert got.kernel_launches == (len(got.route.split(";")) if got.route else 0), (got.kernel_launches, got.route)
        names = [got.col_name(c) for c in range(got.ncols)]
        assert names == list(group_by) + [f"{a.col}_{type(a).__name__.lower()}" for a in aggs]
        for a, agg in enumerate(aggs):
            want = {Sum: L.COL_INT64, Avg: L.COL_DOUBLE, Count: L.COL_COUNT, Min: L.COL_DOUBLE, Max: L.COL_DOUBLE}[type(agg)]
            assert got.col_type(len(group_by) + a) == want
        if n:
            for c in range(got.ncols):
                g = got.column(c)
                assert g.tobytes() == np.asarray(exp[c]).astype(g.dtype).tobytes(), (table, sel, aggs, group_by, c)
            for i in range(min(n, 8)):
                want = []
                for a, agg in enumerate(aggs):
                    v = exp[len(group_by) + a][i]
                    want.append(str(int(v)) if isinstance(agg, (Count, Sum)) else java_double(float(v)))
                assert got.format_row(i) == "Row(" + ",".join(want) + ")"
        return got.route


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg_sum")
    rng = np.random.default_rng(21)
    n = 30_000
    extra = [("mx:DENSE_INT", np.full(n, I32_MAX, np.int32)),
             ("mn:DENSE_INT", np.full(n, I32_MIN, np.int32)),
             ("tn:DENSE_TINYINT", np.full(n, -128, np.int8)),
             ("mix:DENSE_INT", np.where(rng.integers(0, 2, n) == 1, I32_MAX, I32_MIN).astype(np.int32)),
             ("e:PFOR_INT", (np.arange(n) * 70_000).astype(np.int32))]                        # sorted, sums past 2^32
    make_table(d, "t", 50_000, 64, 5, seed=2)                                                # 156 segments
    make_table(d, "neg", 20_000, 32, 10, seed=3, id_mode="random")                          # full int8 / int32 ranges
    make_table(d, "x", n, 1024, 3, seed=4, extra_cols=extra)
    make_table(d, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")       # encoded id: agg_blocks_kernel
    make_table(d, "pr", 20_000, 128, 10, seed=3, id_codec="PFOR_INT", id_mode="random")     # raw mini-blocks, INT_MIN / INT_MAX
    orc, sm = O.Oracle(d), SegmentManager(d)
    yield d, orc, sm
    sm.close()
    orc.close()


SELS = [NoSelect, Select("age", GT(18)), Select("age", EQ(127)), conj(Select("state", Match(["CA", "NY", "DC"])), Select("age", GT(18)))]


def test_every_instantiation(world):
    """NG in {0, 1, 2, 4} x plan NA in {2, 3, 4, 8} on both kernels; the hidden COUNT counts towards NA."""
    d, orc, sm = world
    eng = Engine(sm)
    by_na = {2: [[Sum("age")], [Avg("id"), Count("age")]],
             3: [[Sum("id"), Avg("age")], [Avg("age"), Min("id"), Count("id")]],
             4: [[Avg("age"), Min("id"), Max("age")], [Sum("id"), Count("age"), Max("id"), Avg("id")]],
             8: [[Sum("id"), Avg("age"), Min("id"), Max("age"), Count("id")],
                 [Sum("age"), Sum("id"), Avg("age"), Min("age"), Max("id"), Avg("id"), Min("id")]]}
    for table in ("t", "p"):
        for gb, ng in (([], 0), (["state"], 1), (["state", "age"], 2), (["age", "state", "age"], 4)):
            for na, shapes in by_na.items():
                for aggs in shapes:
                    kern = "agg_blocks" if table == "p" and any(a.col == "id" for a in aggs) else "agg"   # p's id is encoded
                    for sel in SELS[:2]:
                        check_ext(orc, eng, table, sel, aggs, gb, route=f";{kern}<{ng},{na}>/sum;agg_compact")


def test_dense_and_encoded_inputs(world):
    d, orc, sm = world
    eng = Engine(sm)
    for sel in SELS:
        check_ext(orc, eng, "p", sel, [Sum("id"), Avg("id"), Count("id"), Min("id"), Max("id")], ["state"])   # encoded input
        check_ext(orc, eng, "p", sel, [Sum("age"), Avg("age")], ["id"])                                       # encoded group column
        check_ext(orc, eng, "pr", sel, [Sum("id"), Avg("id"), Max("age")], ["state"])
        check_ext(orc, eng, "x", sel, [Sum("e"), Avg("e"), Sum("mx")], ["state"])                             # encoded + dense
        check_ext(orc, eng, "neg", sel, [Sum("id"), Avg("age"), Min("age")], ["state"])


def test_partials_past_32_bits(world):
    """INT_MAX / INT_MIN / TINYINT -128 inputs: a warp's partial leaves 32 bits after a handful of rows."""
    d, orc, sm = world
    eng = Engine(sm)
    for sel in (NoSelect, Select("age", GT(18))):
        for gb in ([], ["state"], ["age"]):
            check_ext(orc, eng, "x", sel, [Sum("mx"), Sum("mn"), Sum("tn"), Avg("mix"), Sum("mix"), Avg("mn")], gb)
    with eng.execute(Query("x", NoSelect, ProjectAgg([Sum("mx"), Sum("mn"), Avg("tn")], [])), sum_avg=True) as r:
        assert r.column(0)[0] == 30_000 * I32_MAX and r.column(1)[0] == 30_000 * I32_MIN and r.column(2)[0] == -128.0


def test_cold_path_and_overflow(world):
    """More than 256 groups per CTA go to the global table row by row; IMM3_AGG_SLOTS = 64 overflows and is reported."""
    d, orc, sm = world
    eng = Engine(sm)
    check_ext(orc, eng, "t", NoSelect, [Sum("age"), Avg("id")], ["id"])                     # 50 000 groups
    check_ext(orc, eng, "p", Select("age", GT(50)), [Avg("age"), Sum("id")], ["id"])
    os.environ["IMM3_AGG_SLOTS"] = "64"
    try:
        for table in ("t", "p"):
            with pytest.raises(Imm3Error) as e:
                eng.execute(Query(table, NoSelect, ProjectAgg([Sum("age")], ["id"])), sum_avg=True)
            assert e.value.status == L.ERR_UNSUPPORTED and "groups" in e.value.message
    finally:
        del os.environ["IMM3_AGG_SLOTS"]


def test_without_sum_avg_equals_imm3_query_agg(world):
    d, orc, sm = world
    eng = Engine(sm)
    shapes = [([Count("id"), Min("age"), Max("id")], ["state"]), ([Min("id")], []), ([Max("age")], ["id"]),
              ([Min("id"), Count("id"), Max("age"), Min("age"), Max("id")], ["state", "age"])]
    for table in ("t", "p", "neg"):
        for sel in SELS:
            for aggs, gb in shapes:
                q = Query(table, sel, ProjectAgg(aggs, gb))
                with eng.execute(q) as a, eng.execute(q, sum_avg=True) as b:
                    assert a.nrows == b.nrows and a.ncols == b.ncols and a.route == b.route
                    for c in range(a.ncols):
                        assert a.col_name(c) == b.col_name(c) and a.col_type(c) == b.col_type(c)
                        assert a.column(c).tobytes() == b.column(c).tobytes()
                    for i in range(min(a.nrows, 5)):
                        assert a.format_row(i) == b.format_row(i)
    for q in (Query("t", NoSelect, ProjectAgg([Min("state")], [])), Query("p", Select("id", GT(5)), ProjectAgg([Min("age")], []))):
        errs = []
        for kw in ({}, {"sum_avg": True}):
            with pytest.raises(Imm3Error) as e:
                eng.execute(q, **kw)
            errs.append((e.value.status, e.value.message))
        assert errs[0] == errs[1]


def test_40m_rows_against_numpy(tmp_path):
    n = 40_000_000
    rng = np.random.default_rng(9)
    v = rng.integers(I32_MIN, I32_MAX, n, dtype=np.int64, endpoint=True).astype(np.int32)
    cols = make_table(tmp_path, "big", n, 1024, 100, seed=3, extra_cols=[("v:DENSE_INT", v)])
    with SegmentManager(str(tmp_path)) as sm:
        eng = Engine(sm)
        for sel, keep in ((Select("age", GT(18)), cols["age"] > 18), (NoSelect, np.ones(n, bool))):
            q = Query("big", sel, ProjectAgg([Sum("v"), Avg("v"), Avg("age"), Sum("id"), Count("id")], ["state"]))
            with eng.execute(q, sum_avg=True) as r:
                st = cols["state"][keep]
                keys, first, inv = np.unique(st, return_index=True, return_inverse=True)
                order = np.argsort(first)
                rank = np.empty_like(order)
                rank[order] = np.arange(len(order))
                g = rank[inv.reshape(-1)]
                cnt = np.bincount(g).astype(np.int64)
                assert list(r.column(0)) == list(keys[order]) and list(r.column(5)) == list(cnt)
                for c, name in ((1, "v"), (4, "id")):
                    s = np.zeros(len(cnt), np.int64)
                    np.add.at(s, g, cols[name][keep].astype(np.int64))
                    assert r.column(c).tolist() == s.tolist()
                    if name == "v":
                        assert r.column(2).tobytes() == (s.astype(np.float64) / cnt.astype(np.float64)).tobytes()
                sa = np.zeros(len(cnt), np.int64)
                np.add.at(sa, g, cols["age"][keep].astype(np.int64))
                assert r.column(3).tobytes() == (sa.astype(np.float64) / cnt.astype(np.float64)).tobytes()


# ---- across ranks -------------------------------------------------------------------------------------------------------

def _cases():
    many = [Sum("id"), Count("id"), Avg("age"), Min("age"), Max("id"), Sum("age"), Avg("id"), Min("id")]
    cases = [("t", Select("age", GT(18)), [Sum("age"), Avg("age")], ["state"]),
             ("t", conj(Select("age", GT(18)), Select("age", LT(30))), [Avg("id"), Count("id"), Max("id")], ["state"]),
             ("t", NoSelect, [Sum("id"), Avg("id")], []),
             ("t", Select("age", EQ(127)), [Sum("age")], ["state"]),                          # nothing matches anywhere
             ("t", conj(Select("id", GT(50000)), Select("id", LT(70000))), [Sum("id"), Avg("age")], ["state"]),
             ("p", NoSelect, [Sum("id"), Avg("id"), Min("id")], []),                         # agg_blocks on every rank
             ("p", Select("age", GT(18)), [Avg("id"), Sum("age")], ["state"]),
             ("p", Select("age", LT(10)), [Sum("age")], ["id"])]                             # encoded group column
    for gb in ([], ["state"], ["state", "age"], ["age", "state", "age"]):
        for na in (1, 2, 3, 7):
            cases.append(("t", Select("age", GT(3)), many[:na], gb))
    return cases


def _worker(rank, world, data_dir, port, out_dir, mode):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch
    import torch.distributed as dist

    import oracle_lib as O
    from agg_sum_ref import query_agg_ext
    from immutable3_b200 import Engine, ProjectAgg, Query, SegmentManager
    from immutable3_b200.dist import CudaExecutor, ShardedEngine, shard_range

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
            for table, sel, aggs, gb in _cases():
                q = Query(table, sel, ProjectAgg(aggs, gb))
                exp = query_agg_ext(whole, table, sel, aggs, gb)
                res = sh.execute_agg(q, sum_avg=True)
                n = len(exp[0]) if len(exp) and len(exp[0]) else 0
                assert res.total == n and len(res.columns) == len(gb) + len(aggs), (rank, table, aggs, gb)
                for c in range(len(res.columns) if n else 0):
                    assert res.columns[c].tobytes() == np.asarray(exp[c]).astype(res.columns[c].dtype).tobytes(), (mode, rank, table, aggs, gb, c)
                # this rank's partials: the same query over its slice of segments
                b, e = shard_range(whole.nsegments(table), rank, world)
                part = query_agg_ext(whole, table, sel, aggs, gb, seg_begin=b, seg_end=e) if e > b else None
                with eng.execute(q, sum_avg=True) as r:
                    pn = len(part[0]) if part is not None and len(part) and len(part[0]) else 0
                    assert r.nrows == pn
                    for c in range(r.ncols if pn else 0):
                        assert r.column(c).tobytes() == np.asarray(part[c]).astype(r.column(c).dtype).tobytes()
                if mode == "device":
                    with eng.execute_agg_global(q, sum_avg=True) as r:
                        assert r.global_count == n
                        assert r.route.endswith("agg_exchange;agg_init;agg_merge;agg_compact"), r.route
                        assert r.kernel_launches == len(r.route.split(";")), (r.kernel_launches, r.route)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def _tables(tmp_path, small=False):
    data = tmp_path / "data"
    if small:
        make_table(data, "t", 600, 64, 5, seed=2)
        make_table(data, "p", 2000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    else:
        make_table(data, "t", 40_000, 64, 5, seed=2)
        make_table(data, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    return data


@pytest.mark.parametrize("world, mode", [(2, "device"), (3, "device"), (2, "host"), (3, "host")])
def test_sharded_sum_avg(tmp_path, world, mode):
    data = _tables(tmp_path)
    port = 41700 + (os.getpid() % 2000) + world + (10 if mode == "host" else 0)
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path), mode), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_sharded_sum_avg_more_ranks_than_segments(tmp_path):
    data = _tables(tmp_path, small=True)
    port = 44700 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(4, str(data), port, str(tmp_path), "device"), nprocs=4, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(4))


def test_global_single_handle_is_local(world):
    d, orc, sm = world
    eng = Engine(sm)
    for table, sel, aggs, gb in _cases():
        if table == "t" or table == "p":
            q = Query(table, sel, ProjectAgg(aggs, gb))
            with eng.execute(q, sum_avg=True) as a, eng.execute_agg_global(q, sum_avg=True) as b:
                assert a.route == b.route and a.nrows == b.nrows
                for c in range(a.ncols):
                    assert a.column(c).tobytes() == b.column(c).tobytes()
