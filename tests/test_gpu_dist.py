"""Segment-sharded execution on real devices, one process per rank.

* host exchange: ShardedEngine over a gloo group, counts all-gathered by torch.distributed (the round-1 path, kept for
  callers without a communicator);
* device exchange: `SegmentManager.comm_connect` - the ranks' GPUs exchange the counts themselves over peer memory
  (imm3_comm_*, k_comm.cuh).  With >= 2 devices every rank has its own GPU and the bootstrap group is NCCL; on a 1-GPU
  box both ranks share cuda:0 (IPC mapping between two processes on one device exercises exactly the same code).

Every rank checks its own slice of the global answer against the oracle run over the WHOLE table.
"""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _cases():
    from helpers import conj
    from immutable3_b200 import EQ, GT, LT, Match, NoSelect, Select

    return [("t", conj(Select("age", GT(18)), Select("age", LT(30))), ["id", "age"]),
            ("t", conj(Select("id", GT(3000)), Select("id", LT(9000))), ["id"]),            # window lands on one rank
            ("t", conj(Select("id", GT(50000)), Select("id", LT(70000))), ["id", "state"]),  # window straddles the rank boundary
            ("t", NoSelect, ["id", "state"]),
            ("t", Select("age", EQ(127)), ["id"]),                                           # nothing matches anywhere
            ("t", conj(Select("state", Match(["CA"])), Select("age", GT(50))), ["state", "age", "id"]),
            ("p", conj(Select("id", GT(2000)), Select("id", LT(900000))), ["id", "age"]),    # sorted-int codec
            ("p", Select("age", LT(10)), ["id"])]


def _worker(rank, world, data_dir, port, out_dir, mode):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch
    import torch.distributed as dist

    import oracle_lib as O
    from helpers import oracle_preds
    from immutable3_b200 import Engine, Project, Query, SegmentManager
    from immutable3_b200.dist import CudaExecutor, ShardedEngine

    ndev = torch.cuda.device_count()
    dev = rank % ndev
    backend = "nccl" if (mode == "device" and ndev >= world) else "gloo"
    if backend == "nccl":
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    os.environ["IMM3_PREFIX_ROWS"] = "8192"  # small tables: let the prefix-first LIMIT policy kick in
    try:
        with SegmentManager(data_dir, device=dev, rank=rank, world=world) as sm, O.Oracle(data_dir) as whole:
            if mode == "device":
                sm.comm_connect()
                assert sm.comm_connected
            eng = ShardedEngine(CudaExecutor(Engine(sm)), collective_device="cuda" if backend == "nccl" else "cpu")
            for table, sel, proj in _cases():
                full = whole.query(table, oracle_preds(sel), proj, limit=0)
                limits = [0, 1, 10, 5000, 10**6]
                if full.nrows > 2:  # cuts right at / around the rank boundary
                    first = eng.execute(Query(table, sel, Project(proj, 0)))
                    limits += [c for c in (first.counts[0] - 1, first.counts[0], first.counts[0] + 1) if c > 0]
                for limit in limits:
                    res = eng.execute(Query(table, sel, Project(proj, limit)))
                    exp = whole.query(table, oracle_preds(sel), proj, limit=limit)
                    assert res.total == exp.nrows, (mode, table, limit, res.counts, res.total, exp.nrows)
                    assert res.take == len(res.columns[0]) if proj else True
                    assert sum(min(c, limit) if limit else c for c in res.counts) >= res.total
                    for c in range(len(proj)):
                        assert np.array_equal(res.columns[c], exp.columns[c][res.offset:res.offset + res.take]), (mode, rank, table, proj[c], limit)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def _tables(tmp_path):
    from helpers import make_table

    data = tmp_path / "data"
    make_table(data, "t", 40_000, 64, 5, seed=2)                                          # 125 segments of 321 rows
    make_table(data, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")  # 10 segments, sorted-int codec
    return data


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_cuda_executor_host_exchange(tmp_path, world):
    data = _tables(tmp_path)
    port = 29700 + (os.getpid() % 2000) + world
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path), "host"), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_cuda_executor_device_exchange(tmp_path, world):
    data = _tables(tmp_path)
    port = 31700 + (os.getpid() % 2000) + world
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path), "device"), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_more_ranks_than_segments_device_exchange(tmp_path):
    """Ranks with an EMPTY slice still take part in every round of the exchange."""
    from helpers import make_table

    data = tmp_path / "data"
    make_table(data, "t", 600, 64, 5, seed=2)    # 2 segments
    make_table(data, "p", 2000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")  # 1 segment
    port = 33700 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(4, str(data), port, str(tmp_path), "device"), nprocs=4, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(4))


def _launches_worker(rank, world, data_dir, port, out_dir):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch.distributed as dist

    import oracle_lib as O
    from helpers import conj, oracle_preds
    from immutable3_b200 import GT, LT, Engine, Project, Query, SegmentManager, Select

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    os.environ["IMM3_COMM_TIMEOUT_MS"] = "10000"
    try:
        with SegmentManager(data_dir, device=0, rank=rank, world=world) as sm, O.Oracle(data_dir) as whole:
            sm.comm_connect()
            eng = Engine(sm)
            for table, sel, proj in [("t", Select("age", LT(50)), ["id", "age"]), ("p", conj(Select("id", GT(2000)), Select("id", LT(900000))), ["id"])]:
                empty = sm.getTable(table).nrows == 0
                for limit in (0, 1, 10, 5000):
                    exp = whole.query(table, oracle_preds(sel), proj, limit=limit)
                    with eng.begin(Query(table, sel, Project(proj, limit))) as h:
                        r = h.route
                        assert h.kernel_launches == (len(r.split(";")) if r else 0), (rank, table, limit, r, h.kernel_launches)
                        assert h.global_count == exp.nrows, (rank, table, limit, h.global_count, exp.nrows, r)
                        if limit:  # rank 0's empty slice fills no LIMIT: every rank runs phase B's exchange round
                            assert r == "count_exchange;count_exchange" if empty else r.endswith(";count_exchange;count_exchange"), (rank, table, limit, r)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_launch_count_matches_the_route_on_small_limits(tmp_path):
    """kernel_launches counts every exchange round of a small LIMIT: rank 0's slice is empty, so its two rounds are all it
    launches, and a rank whose slice is too small for a prefix scans it in phase A and runs phase B's round alone."""
    from helpers import make_table

    data = tmp_path / "data"
    make_table(data, "t", 600, 64, 5, seed=2)    # 2 segments: ranks 1 and 2 own one each
    make_table(data, "p", 2000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")  # 1 segment: rank 2's
    port = 35700 + (os.getpid() % 2000)
    mp.spawn(_launches_worker, args=(3, str(data), port, str(tmp_path)), nprocs=3, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(3))


def test_two_handles_on_two_devices_in_one_process(tmp_path):
    """Kernel attributes (dynamic shared memory limit) are per device: a second handle on another GPU must work."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import oracle_lib as O
    from helpers import conj, make_table, oracle_preds
    from immutable3_b200 import GT, LT, Engine, Project, Query, SegmentManager, Select

    data = tmp_path / "data"
    make_table(data, "t", 40_000, 64, 5, seed=2)
    make_table(data, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    with O.Oracle(str(data)) as orc, SegmentManager(str(data), device=0) as a, SegmentManager(str(data), device=1) as b:
        for table, sel, proj in [("t", conj(Select("age", GT(18)), Select("age", LT(30))), ["id", "age"]),
                                 ("p", conj(Select("id", GT(2000)), Select("id", LT(900000))), ["id", "age"])]:
            exp = orc.query(table, oracle_preds(sel), proj, limit=0)
            for sm in (b, a, b):
                with Engine(sm).execute(Query(table, sel, Project(proj, 0))) as got:
                    assert got.nrows == exp.nrows
                    for c in range(len(proj)):
                        assert np.array_equal(got.column(c), exp.columns[c])
