"""ShardedEngine.execute_agg without a communicator, on CPU: world-size 2 and 3 gloo groups all-gather every rank's
partial groups and merge them on the host in rank order.  The local executor is backed by the ORACLE over the rank's
canonical slice (there is no GPU here and the product has no CPU path); every rank must end up with the oracle's answer
over the WHOLE table - group order, keys, counts and extremes.  Also: the GPU entry point refuses an unconnected
sharded handle before any device work."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))


class OracleAggExecutor:
    """begin / finish of a ProjectAgg query over the oracle restricted to this rank's canonical slice (its partials)."""

    def __init__(self, data_dir, rank, world):
        import oracle_lib as O
        from immutable3_b200.dist import shard_range

        self.orc = O.Oracle(data_dir)
        self.rank, self.world = rank, world
        self.shard_range = shard_range

    def begin(self, query):
        from helpers import oracle_preds

        a, b = self.shard_range(self.orc.nsegments(query.table), self.rank, self.world)
        r = self.orc.query_agg(query.table, oracle_preds(query.select), _oracle_aggs(query.project.aggs), list(query.project.groupBy),
                               seg_begin=a, seg_end=b)
        r.local_count = r.nrows
        return r

    def finish(self, handle, take):
        return [np.asarray(c)[:take] for c in handle.columns]


def _oracle_aggs(aggs):
    import oracle_lib as O
    from immutable3_b200 import Count, Max, Min

    ops = {Count: O.AGG_COUNT, Min: O.AGG_MIN, Max: O.AGG_MAX}
    return [(ops[type(a)], a.col) for a in aggs]


def _cases():
    from helpers import conj
    from immutable3_b200 import EQ, GT, LT, Count, Match, Max, Min, NoSelect, Select

    mm = [Min("age"), Max("age")]
    return [(Select("age", GT(18)), mm, ["state"]),                                     # the reference's example
            (conj(Select("age", GT(18)), Select("age", LT(40))), [Count("id"), Min("id"), Max("id")], ["age"]),  # keys first seen on later ranks
            (NoSelect, [Count("state"), Max("id")], ["state", "age"]),
            (NoSelect, [Count("id"), Min("id"), Max("age")], []),                       # no group-by: one row
            (Select("age", EQ(127)), mm, ["state"]),                                    # empty everywhere
            (conj(Select("id", GT(300)), Select("id", LT(360))), [Count("id"), Min("age")], ["state"]),  # groups on one rank only
            (conj(Select("id", GT(300)), Select("id", LT(360))), [Max("id")], []),
            (conj(Select("state", Match(["CA", "NY"])), Select("age", GT(50))), [Count("id"), Max("age"), Min("id")], ["state"])]


def _worker(rank, world, data_dir, port, out_dir):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch.distributed as dist

    import oracle_lib as O
    from helpers import oracle_preds
    from immutable3_b200 import ProjectAgg, Query
    from immutable3_b200.dist import ShardedEngine

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        ex = OracleAggExecutor(data_dir, rank, world)
        eng = ShardedEngine(ex)
        whole = O.Oracle(data_dir)
        saw_late_key = saw_idle_rank = False
        for sel, aggs, gb in _cases():
            q = Query("t", sel, ProjectAgg(aggs, gb))
            res = eng.execute_agg(q)
            exp = whole.query_agg("t", oracle_preds(sel), _oracle_aggs(aggs), gb)
            assert res.total == res.take == exp.nrows and res.offset == 0, (sel, aggs, gb, res.counts, exp.nrows)
            assert len(res.counts) == world
            assert res.counts[rank] == ex.begin(q).nrows
            assert len(res.columns) == len(gb) + len(aggs)
            for c in range(len(res.columns)):
                assert res.columns[c].dtype == np.asarray(exp.columns[c]).dtype, (sel, c)
                assert np.array_equal(res.columns[c], np.asarray(exp.columns[c])), (rank, sel, aggs, gb, c)
            if gb and res.counts[0] < exp.nrows and exp.nrows > 0:
                saw_late_key = True        # a group the first rank does not hold
            if exp.nrows > 0 and 0 in res.counts:
                saw_idle_rank = True       # a rank that contributes no group
        assert saw_late_key and saw_idle_rank
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_agg_over_gloo(tmp_path, world):
    from helpers import make_table

    data = tmp_path / "data"
    make_table(data, "t", 13 * (8 * 2 + 1) + 5, 8, 2, seed=2)  # 14 segments: lexicographic canonical order
    port = 30500 + (os.getpid() % 2000) + world
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_merge_partials_rank_order():
    """The first rank that holds a key decides its position; Count adds up, Min / Max take the extreme."""
    from immutable3_b200 import Count, Max, Min
    from immutable3_b200.dist import merge_partials

    s = lambda *v: np.array(v, dtype="S2")
    parts = [[s("CA", "NY"), np.array([2, 1], np.int64), np.array([5.0, 7.0]), np.array([9.0, 7.0])],
             [s(), np.array([], np.int64), np.array([]), np.array([])],
             [s("TX", "CA"), np.array([4, 3], np.int64), np.array([1.0, -2.0]), np.array([1.0, 11.0])]]
    cols = merge_partials(parts, 1, [Count("id"), Min("age"), Max("age")])
    assert list(cols[0]) == [b"CA", b"NY", b"TX"]
    assert list(cols[1]) == [5, 1, 4] and cols[1].dtype == np.int64
    assert list(cols[2]) == [-2.0, 7.0, 1.0] and list(cols[3]) == [11.0, 7.0, 1.0]
    empty = merge_partials([[s(), np.array([], np.int64)]] * 2, 1, [Count("id")])
    assert len(empty) == 2 and len(empty[0]) == 0 and empty[0].dtype == np.dtype("S2")


def test_global_agg_refuses_unconnected_sharded_handle(tmp_path):
    from helpers import make_table
    from immutable3_b200 import Engine, GT, Imm3Error, Max, Min, ProjectAgg, Query, SegmentManager, Select
    from immutable3_b200 import _lib as L

    make_table(tmp_path, "t", 600, 64, 5, seed=2)
    q = Query("t", Select("age", GT(18)), ProjectAgg([Min("age"), Max("age")], ["state"]))
    with SegmentManager(str(tmp_path), rank=1, world=2, flags=L.OPEN_HOST_ONLY) as sm:
        with pytest.raises(Imm3Error) as e:
            Engine(sm).execute_agg_global(q)
        assert e.value.status == L.ERR_STATE
        assert "imm3_comm_connect" in e.value.message
