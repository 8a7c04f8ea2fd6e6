"""count / min / max ... group by with sorted-int-codec (PFOR_INT) columns as MIN / MAX inputs and group columns
(agg_blocks_kernel: the encoded columns decoded block by block inside the aggregation) against the oracle, against the same
rows stored with a dense id, and against numpy at 40 M rows."""
import numpy as np
import pytest

import oracle_lib as O
from helpers import conj, make_table, oracle_preds
from test_gpu_agg import _OPS, check_agg
from immutable3_b200 import Count, EQ, Engine, GT, Imm3Error, Match, Max, Min, NoSelect, ProjectAgg, Query, SegmentManager, Select
from immutable3_b200 import _lib as L

pytestmark = pytest.mark.gpu

SELS = [NoSelect, Select("age", GT(18)), Select("age", EQ(127)), conj(Select("state", Match(["CA", "NY", "DC"])), Select("age", GT(18)))]


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg_enc")
    rng = np.random.default_rng(5)
    n = 30_000
    extra = [("day:PFOR_INT", (np.arange(n) // 1500).astype(np.int32)),                       # sorted, 20 values
             ("seq:PFOR_INT", (np.arange(n) + 7).astype(np.int32)),                           # strictly sorted: the dense shape
             ("e3:PFOR_INT", np.cumsum(rng.integers(0, 5000, n)).astype(np.int32))]           # sorted, irregular widths
    make_table(d, "p", n, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps", extra_cols=extra)
    make_table(d, "pr", 20_000, 128, 10, seed=3, id_codec="PFOR_INT", id_mode="random")      # raw 32-bit mini-blocks, INT_MIN / INT_MAX
    make_table(d, "rag", 12_001, 100, 3, seed=2, id_codec="PFOR_INT", id_mode="steps")       # 41 segments, a 1-row tail block
    make_table(d, "one", 1, 8, 2, seed=2, id_codec="PFOR_INT")
    make_table(d, "tp", 50_000, 1024, 7, seed=6, id_codec="PFOR_INT", id_mode="steps")        # twins: same rows, encoded / dense id
    make_table(d, "td", 50_000, 1024, 7, seed=6, id_codec="DENSE_INT", id_mode="steps")
    orc, sm = O.Oracle(d), SegmentManager(d)
    yield d, orc, sm
    sm.close()
    orc.close()


def test_encoded_aggregates_match_the_oracle(world):
    d, orc, sm = world
    eng = Engine(sm)
    shapes = [([Min("id"), Max("id")], []),
              ([Count("id"), Min("id"), Max("id")], ["state"]),
              ([Count("age")], ["id"]),                                       # encoded column as the only group column
              ([Max("age"), Min("id")], ["id", "state", "age"]),              # 4 + 2 + 1 key bytes
              ([Min("id"), Max("id"), Count("age")], ["id"])]                 # the same encoded column as group and aggregate
    total = 0
    for table in ("p", "pr", "rag"):
        for sel in SELS:
            for aggs, gb in shapes:
                total += check_agg(orc, eng, table, sel, aggs, gb)
    assert total > 10_000
    for sel in SELS:
        check_agg(orc, eng, "p", sel, [Count("age")], ["day"])                                # low-cardinality sorted key
        check_agg(orc, eng, "p", sel, [Min("seq"), Max("seq"), Max("id")], ["state"])         # two encoded columns, dense shape
        check_agg(orc, eng, "p", sel, [Min("id"), Max("seq"), Min("day")], ["e3"])            # four distinct encoded columns
    check_agg(orc, eng, "one", NoSelect, [Min("id"), Max("id"), Count("age")], ["id"])
    check_agg(orc, eng, "one", Select("age", EQ(127)), [Min("id")], ["state"])


def test_every_instantiation(world):
    """agg_blocks_kernel<NG, NA>: 0 / 1 / 2 / "up to 4" group columns x 1 .. 4 / "up to 8" aggregates, an encoded column in each."""
    d, orc, sm = world
    eng = Engine(sm)
    many = [Min("id"), Count("id"), Max("seq"), Min("age"), Max("age"), Count("state"), Max("id"), Min("day")]
    for gb in ([], ["state"], ["state", "age"], ["day", "state", "age"], ["age", "state", "age", "state"]):
        for na in (1, 2, 3, 4, 5, 8):
            check_agg(orc, eng, "p", Select("age", GT(3)), many[:na], gb)
            check_agg(orc, eng, "p", Select("age", EQ(5)), [Max("seq")] + many[8 - na + 1:], gb)   # sparse selection


def test_encoded_and_dense_twins_agree(world):
    d, orc, sm = world
    eng = Engine(sm)
    for sel in SELS + [Select("state", Match(["CA"]))]:
        for aggs, gb in (([Count("id"), Min("id"), Max("id")], ["state"]), ([Min("id"), Max("id")], ["age"]),
                         ([Min("id"), Max("id"), Count("age")], []), ([Count("age"), Max("age")], ["id", "state"])):
            with eng.execute(Query("tp", sel, ProjectAgg(aggs, gb))) as a, eng.execute(Query("td", sel, ProjectAgg(aggs, gb))) as b:
                assert a.nrows == b.nrows and a.ncols == b.ncols
                for c in range(a.ncols):
                    assert a.col_name(c) == b.col_name(c) and np.array_equal(a.column(c), b.column(c)), (sel, aggs, gb, c)


def test_overflow_and_errors(world, monkeypatch):
    d, orc, sm = world
    eng = Engine(sm)
    assert check_agg(orc, eng, "p", NoSelect, [Count("age"), Min("id")], ["seq"]) == 30_000   # > 256 groups per CTA: the global table
    monkeypatch.setenv("IMM3_AGG_SLOTS", "64")
    with pytest.raises(Imm3Error) as e:
        eng.execute(Query("p", NoSelect, ProjectAgg([Min("id")], ["seq"])))
    assert e.value.status == L.ERR_UNSUPPORTED                                                # reported, not truncated
    monkeypatch.delenv("IMM3_AGG_SLOTS")
    check_agg(orc, eng, "p", Select("age", GT(18)), [Min("id"), Max("id")], ["state"])         # the handle is fine afterwards
    with pytest.raises(Imm3Error) as e:
        eng.execute(Query("p", Select("id", GT(5)), ProjectAgg([Min("id")], [])))
    assert e.value.status == L.ERR_UNSUPPORTED                                                # predicates on the encoded column


def test_sharded_partials_merge_to_the_whole(world):
    d, orc, sm = world
    aggs, gb = [Count("age"), Min("id"), Max("id")], ["state"]
    sel = Select("age", GT(40))
    exp = orc.query_agg("rag", oracle_preds(sel), [(_OPS[type(a)], a.col) for a in aggs], gb)
    for world_size in (2, 3, 8):
        merged, order = {}, []
        for rank in range(world_size):
            with SegmentManager(d, rank=rank, world=world_size) as part:
                with Engine(part).execute(Query("rag", sel, ProjectAgg(aggs, gb))) as r:
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


def _numpy_group(keys, mask, vals):
    """First-appearance order of the selected keys, and count / min / max of vals per key."""
    k, v = keys[mask], vals[mask]
    uniq, first, inv = np.unique(k, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")
    cnt = np.bincount(inv, minlength=len(uniq))
    mn = np.full(len(uniq), np.iinfo(np.int64).max)
    mx = np.full(len(uniq), np.iinfo(np.int64).min)
    np.minimum.at(mn, inv, v.astype(np.int64))
    np.maximum.at(mx, inv, v.astype(np.int64))
    return uniq[order], cnt[order], mn[order], mx[order]


def test_40m_rows_against_numpy(tmp_path):
    from immutable3_b200.loader import synth_write

    n = 40_000_000
    synth_write(str(tmp_path), "t", n, 1024, 1000, L.CODEC_PFOR_INT)
    with O.Oracle(tmp_path) as orc:
        raw = orc.query("t", [], ["id", "state", "age"])                 # the segment files, decoded in canonical order
    ids, states, ages = (np.asarray(c) for c in raw.columns)
    assert len(ids) == n
    with SegmentManager(tmp_path) as sm:
        eng = Engine(sm)
        keys, cnt, mn, mx = _numpy_group(states, ages > 18, ids)       # Q1
        with eng.execute(Query("t", Select("age", GT(18)), ProjectAgg([Count("id"), Min("id"), Max("id")], ["state"]))) as r:
            assert np.array_equal(r.column(0), keys) and np.array_equal(r.column(1), cnt)
            assert np.array_equal(r.column(2), mn.astype(np.float64)) and np.array_equal(r.column(3), mx.astype(np.float64))
        keys, cnt, mn, mx = _numpy_group(ages, states == b"CA", ids)   # Q2
        with eng.execute(Query("t", Select("state", Match(["CA"])), ProjectAgg([Min("id"), Max("id")], ["age"]))) as r:
            assert np.array_equal(r.column(0), keys)
            assert np.array_equal(r.column(1), mn.astype(np.float64)) and np.array_equal(r.column(2), mx.astype(np.float64))
