"""count / min / max ... group by on the GPU (imm3_query_agg, k_agg.cuh) against the oracle's restatement of ProjectAggOp /
ProjectAggregateQueueOp: same groups, same order (first appearance in canonical row order), same values, same printed rows."""
import os

import numpy as np
import pytest

import oracle_lib as O
from helpers import conj, make_table, oracle_preds
from immutable3_b200 import (Avg, Count, EQ, Engine, GT, Imm3Error, LT, Match, Max, Min, NoSelect, ProjectAgg, Query, SegmentManager, Select,
                             Sum)
from immutable3_b200 import _lib as L

pytestmark = pytest.mark.gpu
_OPS = {Count: O.AGG_COUNT, Min: O.AGG_MIN, Max: O.AGG_MAX}


def _java_double(v):
    if v == 0:
        return "0.0"
    a = abs(int(v))
    s = str(a)
    if a < 10_000_000:
        return ("-" if v < 0 else "") + s + ".0"
    frac = s[1:].rstrip("0") or "0"
    return ("-" if v < 0 else "") + s[0] + "." + frac + "E" + str(len(s) - 1)


def check_agg(orc, eng, table, sel, aggs, group_by):
    exp = orc.query_agg(table, oracle_preds(sel), [(_OPS[type(a)], a.col) for a in aggs], list(group_by))
    with eng.execute(Query(table, sel, ProjectAgg(aggs, group_by))) as got:
        assert got.nrows == exp.nrows, (table, sel, aggs, group_by, got.nrows, exp.nrows)
        assert got.ncols == len(group_by) + len(aggs)
        for c in range(got.ncols):
            assert got.col_type(c) == exp.types[c]
            assert np.array_equal(got.column(c), exp.columns[c]), (table, sel, aggs, group_by, c)
        for i in range(min(got.nrows, 20)):   # Row(repr, repr, ...): the aggregators only (ProjectAggregateQueue.scala:48-50)
            want = "Row(" + ",".join(str(int(exp.columns[len(group_by) + a][i])) if isinstance(aggs[a], Count) else _java_double(exp.columns[len(group_by) + a][i])
                                     for a in range(len(aggs))) + ")"
            assert got.format_row(i) == want
        names = [got.col_name(c) for c in range(got.ncols)]
        assert names == list(group_by) + [f"{a.col}_{type(a).__name__.lower()}" for a in aggs]
        assert got.kernel_launches == (len(got.route.split(";")) if got.route else 0), (got.kernel_launches, got.route)
        return got.nrows


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg")
    rng = np.random.default_rng(11)
    make_table(d, "t", 50_000, 64, 5, seed=2)                          # 156 segments: lexicographic canonical order
    make_table(d, "neg", 20_000, 32, 10, seed=3, id_mode="random")     # full int8 / int32 ranges
    n = 30_000
    extra = [("zip:DENSE_STRING:size=4", np.array([b"1234", b"9876", b"0000"], "S4")[rng.integers(0, 3, n)]),
             ("big:DENSE_INT", (rng.integers(0, 3, n) * 1_000_000_000 - 1_000_000_000 + rng.integers(0, 5, n)).astype(np.int32))]
    make_table(d, "wide", n, 100, 7, seed=8, extra_cols=extra)
    make_table(d, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    make_table(d, "one", 1, 8, 2, seed=2)
    orc, sm = O.Oracle(d), SegmentManager(d)
    yield d, orc, sm
    sm.close()
    orc.close()


def test_aggregates_match_the_oracle(world):
    d, orc, sm = world
    eng = Engine(sm)
    sels = [NoSelect, Select("age", GT(18)), conj(Select("age", GT(18)), Select("age", LT(30))), Select("age", EQ(127)),
            conj(Select("state", Match(["CA", "NY", "DC"])), Select("id", GT(1000)))]
    shapes = [([Min("age"), Max("age")], ["state"]),                      # the reference's own example (Engine.scala:66-78)
              ([Count("state")], []), ([Count("id"), Min("id"), Max("id")], ["age"]), ([Max("id"), Count("age")], ["state", "age"]),
              ([Min("age")], ["age", "state"]), ([Count("age"), Count("id")], ["state"])]
    total = 0
    for table in ("t", "neg"):
        for sel in sels:
            for aggs, gb in shapes:
                total += check_agg(orc, eng, table, sel, aggs, gb)
    assert total > 1000
    check_agg(orc, eng, "wide", Select("age", LT(50)), [Min("big"), Max("big"), Count("zip")], ["zip"])   # doubles beyond 10^7: "1.000000004E9"
    check_agg(orc, eng, "wide", NoSelect, [Max("big")], ["zip", "state"])                                 # 6 key bytes
    check_agg(orc, eng, "one", NoSelect, [Count("id"), Min("age")], ["state"])
    check_agg(orc, eng, "p", Select("age", GT(90)), [Count("age"), Max("age")], ["state"])                # encoded table, dense predicate
    check_agg(orc, eng, "t", NoSelect, [Count("id")], ["id"])                                             # 50 000 groups: the CTA tables overflow
    # every instantiation of agg_kernel<NG, NA>: 0 / 1 / 2 / "up to 4" group-by columns x 1 .. 4 / "up to 8" aggregates
    many = [Count("id"), Min("id"), Max("id"), Min("age"), Max("age"), Count("state"), Max("big"), Min("big")]
    for gb in ([], ["state"], ["state", "age"], ["zip", "state", "age"], ["age", "state", "age", "state"]):
        for na in (1, 2, 3, 4, 5, 8):
            check_agg(orc, eng, "wide", Select("age", GT(3)), many[:na], gb)
            check_agg(orc, eng, "wide", Select("age", EQ(5)), many[8 - na:], gb)                          # sparse selection, MIN / MAX first


def test_aggregate_errors_are_status_codes(world, monkeypatch):
    d, orc, sm = world
    eng = Engine(sm)

    def status(q):
        with pytest.raises(Imm3Error) as e:
            eng.execute(q)
        return e.value.status

    assert status(Query("t", NoSelect, ProjectAgg([Sum("age")], []))) == L.ERR_UNSUPPORTED      # Engine.scala:153
    assert status(Query("t", NoSelect, ProjectAgg([Avg("age")], []))) == L.ERR_UNSUPPORTED
    assert status(Query("t", NoSelect, ProjectAgg([Min("state")], []))) == L.ERR_UNSUPPORTED    # Engine.scala:147
    assert status(Query("t", NoSelect, ProjectAgg([Min("nope")], []))) == L.ERR_NOT_FOUND
    assert status(Query("t", NoSelect, ProjectAgg([Min("age")], ["nope"]))) == L.ERR_NOT_FOUND
    assert status(Query("nope", NoSelect, ProjectAgg([Min("age")], []))) == L.ERR_NOT_FOUND
    assert status(Query("t", NoSelect, ProjectAgg([Count("age")], ["id", "id"]))) == L.ERR_UNSUPPORTED  # 8 key bytes
    assert status(Query("p", Select("id", GT(5)), ProjectAgg([Count("age")], []))) == L.ERR_UNSUPPORTED
    assert status(Query("t", Select("state", GT(5)), ProjectAgg([Count("age")], []))) == L.ERR_UNSUPPORTED  # Select.scala:80
    monkeypatch.setenv("IMM3_AGG_SLOTS", "64")
    assert status(Query("t", NoSelect, ProjectAgg([Count("id")], ["id"]))) == L.ERR_UNSUPPORTED  # more groups than table slots: reported, not truncated
    monkeypatch.delenv("IMM3_AGG_SLOTS")
    check_agg(orc, eng, "t", Select("age", GT(18)), [Min("age"), Max("age")], ["state"])             # the handle is fine afterwards


def test_sharded_partials_merge_to_the_whole(world):
    """Per-rank partial aggregates merged in rank order (count: sum, min / max: min / max, group order: first appearance) =
    the aggregate of the whole table - what ProjectAggregateQueueOp does with the per-segment maps."""
    d, orc, sm = world
    aggs, gb = [Count("age"), Min("id"), Max("age")], ["state"]
    sel = Select("age", GT(40))
    exp = orc.query_agg("t", oracle_preds(sel), [(_OPS[type(a)], a.col) for a in aggs], gb)
    for world_size in (2, 3, 8):
        merged, order = {}, []
        for rank in range(world_size):
            with SegmentManager(d, rank=rank, world=world_size) as part:
                with Engine(part).execute(Query("t", sel, ProjectAgg(aggs, gb))) as r:
                    cols = r.columns()
                    for i in range(r.nrows):
                        k = cols[0][i]
                        if k not in merged:
                            merged[k] = [0, np.inf, -np.inf]
                            order.append(k)
                        m = merged[k]
                        m[0] += int(cols[1][i])
                        m[1] = min(m[1], float(cols[2][i]))
                        m[2] = max(m[2], float(cols[3][i]))
        assert order == list(exp.columns[0])
        assert [merged[k][0] for k in order] == list(exp.columns[1])
        assert [merged[k][1] for k in order] == list(exp.columns[2]) and [merged[k][2] for k in order] == list(exp.columns[3])
