"""Global aggregates across segment-sharded ranks (imm3_query_agg_global, ShardedEngine.execute_agg), one process per rank.

* device exchange: `SegmentManager.comm_connect`, then every rank's GPU merges all ranks' partial groups itself
  (k_comm.cuh agg_exchange_kernel, k_agg.cuh agg_merge_kernel).  With >= `world` devices every rank has its own GPU and
  the bootstrap group is NCCL; on a 1-GPU box the ranks share cuda:0 through IPC (the same code path).
* host exchange: ShardedEngine.execute_agg over gloo without a communicator (partials all-gathered, merged on the host).

Every rank's result must equal the oracle's query_agg over the WHOLE table: group order, keys, counts and extremes.
"""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
SEG_ROWS = 5 * 64 + 1  # rows of a full segment of the "g" table (segment_size 5, blocks of 64)


def _cases():
    from helpers import conj
    from immutable3_b200 import EQ, GT, LT, Count, Match, Max, Min, NoSelect, Select

    mm = [Min("age"), Max("age")]
    many = [Min("id"), Count("id"), Max("age"), Min("age"), Max("id"), Count("state"), Max("age"), Min("id")]
    cases = [("t", Select("age", GT(18)), mm, ["state"]),                                     # the reference's example
             ("t", conj(Select("age", GT(18)), Select("age", LT(30))), [Count("id"), Min("id"), Max("id")], ["state"]),
             ("t", conj(Select("age", GT(60)), Select("age", LT(90))), [Count("id"), Max("id")], ["age"]),
             ("t", NoSelect, [Count("id"), Min("id"), Max("age")], []),                       # no group-by
             ("t", Select("age", EQ(127)), mm, ["state"]),                                    # nothing matches anywhere
             ("t", conj(Select("id", GT(3000)), Select("id", LT(9000))), [Count("id"), Min("age")], ["state"]),    # one rank
             ("t", conj(Select("id", GT(50000)), Select("id", LT(70000))), [Count("id"), Max("id")], ["state"]),  # straddles
             ("t", conj(Select("state", Match(["CA", "NY"])), Select("age", GT(50))), [Max("id"), Min("id")], ["state", "age"]),
             ("p", NoSelect, [Min("id"), Max("id")], []),                                     # agg_blocks on every rank
             ("p", Select("age", GT(18)), [Count("id"), Min("id"), Max("id")], ["state"]),
             ("p", Select("age", LT(10)), [Count("age")], ["id"]),                            # encoded group column
             ("p", NoSelect, [Max("age"), Min("id")], ["id", "state", "age"])]
    for gb in ([], ["state"], ["state", "age"], ["age", "state", "age"]):                   # the NG x NA instantiations
        for na in (1, 2, 3, 4, 5, 8):
            cases.append(("t", Select("age", GT(3)), many[:na], gb))
    return cases


def _oracle(orc, table, sel, aggs, gb):
    import oracle_lib as O
    from helpers import oracle_preds
    from immutable3_b200 import Count, Max, Min

    ops = {Count: O.AGG_COUNT, Min: O.AGG_MIN, Max: O.AGG_MAX}
    return orc.query_agg(table, oracle_preds(sel), [(ops[type(a)], a.col) for a in aggs], list(gb))


def _same(cols, exp, what):
    assert len(cols) == len(exp.columns), what
    assert (len(cols[0]) if cols else 0) == exp.nrows, (what, len(cols[0]), exp.nrows)
    for c in range(len(cols)):
        assert np.array_equal(cols[c], np.asarray(exp.columns[c])), (what, c)


def _worker(rank, world, data_dir, port, out_dir, mode):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch
    import torch.distributed as dist

    import oracle_lib as O
    from helpers import conj
    from immutable3_b200 import Count, Engine, GT, Imm3Error, LT, Max, Min, NoSelect, Project, ProjectAgg, Query, SegmentManager, Select
    from immutable3_b200 import _lib as L
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

            def check_global(table, sel, aggs, gb):
                q = Query(table, sel, ProjectAgg(aggs, gb))
                exp = _oracle(whole, table, sel, aggs, gb)
                res = sh.execute_agg(q)
                _same(res.columns, exp, (mode, rank, table, sel, aggs, gb))
                assert res.offset == 0 and res.take == res.total == exp.nrows and len(res.counts) == world
                with eng.execute(q) as part:  # this rank's partials (imm3_query_agg is unchanged)
                    assert res.counts[rank] == part.nrows
                if mode == "device":
                    with eng.execute_agg_global(q) as r:
                        _same(r.columns(), exp, (rank, table, sel, aggs, gb))
                        assert r.global_count == exp.nrows and r.rank_counts == res.counts
                        assert r.route.endswith("agg_exchange;agg_init;agg_merge;agg_compact"), r.route
                        assert r.kernel_launches == len(r.route.split(";")), (r.kernel_launches, r.route)
                return res

            for table, sel, aggs, gb in _cases():
                check_global(table, sel, aggs, gb)

            if mode == "device":
                # one rank's slice overflows its table: the error bit reaches every rank, nobody times out
                os.environ["IMM3_AGG_SLOTS"] = "64"
                for q in (Query("g", NoSelect, ProjectAgg([Count("id")], ["h"])),      # > 64 groups on rank 0 only
                          Query("g", NoSelect, ProjectAgg([Min("id")], ["g"]))):        # <= 64 per rank, > 64 merged
                    with pytest.raises(Imm3Error) as e:
                        eng.execute_agg_global(q)
                    assert e.value.status == L.ERR_UNSUPPORTED, e.value.message
                os.environ["IMM3_AGG_SLOTS"] = "131072"                                # above the exchange buffer
                with pytest.raises(Imm3Error) as e:
                    eng.execute_agg_global(Query("g", NoSelect, ProjectAgg([Min("id")], ["g"])))
                assert e.value.status == L.ERR_UNSUPPORTED
                del os.environ["IMM3_AGG_SLOTS"]
                check_global("g", NoSelect, [Count("id"), Min("id")], ["h"])           # the handles answer correctly afterwards
                check_global("g", NoSelect, [Min("id"), Max("id")], ["g"])

            # back-to-back aggregates with changing group sets, interleaved with Project queries on the count exchange:
            # a stale exchange buffer or a broken memory ordering shows up as a wrong group
            for i in range(44):
                hi = 7 + (i * 37) % 100
                check_global("g", Select("g", LT(hi)), [Count("id"), Min("id"), Max("id")] if i % 2 else [Max("age")], ["g"] if i % 3 else ["g", "state"])
                if i % 4 == 0:
                    sel = conj(Select("g", GT(hi // 2)), Select("g", LT(hi)))
                    res = sh.execute(Query("g", sel, Project(["id"], 0)))
                    exp = whole.query("g", [("g", O.OP_GT, hi // 2), ("g", O.OP_LT, hi)], ["id"], limit=0)
                    assert res.total == exp.nrows
                    assert np.array_equal(res.columns[0], np.asarray(exp.columns[0])[res.offset:res.offset + res.take])
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def _tables(tmp_path, small=False):
    from helpers import make_table

    data = tmp_path / "data"
    if small:  # fewer segments than ranks: some ranks hold nothing
        make_table(data, "t", 600, 64, 5, seed=2)                                            # 2 segments
        make_table(data, "p", 2000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")   # 1 segment
    else:
        make_table(data, "t", 40_000, 64, 5, seed=2)                                         # 125 segments of 321 rows
        make_table(data, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    # "g": 10 segments (canonical order = write order): g = 10 distinct values per segment, disjoint across segments;
    # h = 100 distinct values in segment 0, one value elsewhere
    n = 10 * SEG_ROWS
    row = np.arange(n)
    seg = row // SEG_ROWS
    g = (seg * 10 + row % 10).astype(np.int32)
    h = np.where(seg == 0, row % 100, 1000).astype(np.int32)
    make_table(data, "g", n, 64, 5, seed=6, extra_cols=[("g:DENSE_INT", g), ("h:DENSE_INT", h)])
    return data


@pytest.mark.parametrize("world", [2, 3])
def test_global_agg_device_exchange(tmp_path, world):
    data = _tables(tmp_path)
    port = 35700 + (os.getpid() % 2000) + world
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path), "device"), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


@pytest.mark.parametrize("world", [2, 3])
def test_global_agg_host_exchange(tmp_path, world):
    data = _tables(tmp_path)
    port = 37700 + (os.getpid() % 2000) + world
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path), "host"), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_global_agg_more_ranks_than_segments(tmp_path):
    """Ranks with an EMPTY slice take part in every exchange with 0 groups."""
    data = _tables(tmp_path, small=True)
    port = 39700 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(4, str(data), port, str(tmp_path), "device"), nprocs=4, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(4))


def test_global_agg_single_handle_is_imm3_query_agg(tmp_path):
    """world == 1: imm3_query_agg_global returns exactly what imm3_query_agg returns, route included."""
    sys.path.insert(0, HERE)
    from immutable3_b200 import Engine, ProjectAgg, Query, SegmentManager

    data = _tables(tmp_path)
    with SegmentManager(str(data)) as sm:
        eng = Engine(sm)
        for table, sel, aggs, gb in _cases():
            q = Query(table, sel, ProjectAgg(aggs, gb))
            with eng.execute(q) as a, eng.execute_agg_global(q) as b:
                assert a.nrows == b.nrows and a.ncols == b.ncols and a.route == b.route
                assert b.rank_counts == a.rank_counts and b.global_count == a.global_count == b.nrows
                assert "agg_exchange" not in b.route
                for c in range(a.ncols):
                    assert a.col_name(c) == b.col_name(c) and np.array_equal(a.column(c), b.column(c))
