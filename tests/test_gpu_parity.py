"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle, bit-exact, on the
same tables and queries — rows, values and order (SURVEY.md §3.4-8).  Every test needs a GPU."""
import os
import re

import numpy as np
import pytest

import oracle_lib as O
from helpers import STATES, conj, make_table, oracle_preds
from immutable3_b200 import (And, EQ, Engine, GT, Imm3Error, LT, Match, NoSelect, OPEN_FORCE_BLOCKS, OPEN_KEEP_HOST, OPEN_NO_TMA,
                             Or, Project, Query, SegmentManager, Select)
from immutable3_b200 import _lib as L
from immutable3_b200.dist import limit_split
from immutable3_b200.loader import synth_write

pytestmark = pytest.mark.gpu

# variant -> (imm3_open flags, IMM3_PATH): the single-pass block kernel forced onto dense tables (IMM3_PATH=fused selects it
# on block tables), the block pipeline forced onto dense tables (row-space filter kernel -> block emit kernel) with TMA staging /
# direct loads, the dense multi-pass pipeline (filter -> offset scan -> emit: what the library picks for a dense table) with TMA
# staging / direct loads, and the library's own choice.  On the dense tables below "multi" is the same configuration as "auto";
# it also checks from the route that the multi-pass kernels ran, and "multi_direct" that no TMA kernel did (ROUTE_CHECKS).
VARIANT_DEFS = {"blocks": (OPEN_FORCE_BLOCKS, "fused"), "blocks_multi": (OPEN_FORCE_BLOCKS, ""), "blocks_no_tma": (OPEN_FORCE_BLOCKS | OPEN_NO_TMA, ""),
                "multi": (0, ""), "multi_direct": (OPEN_NO_TMA, ""), "auto": (0, "")}
ROUTE_CHECKS = {"multi": r"^(?!.*(blocks_|scan_blocks))", "multi_direct": r"^(?!.*(blocks_|scan_blocks|filter\(tma\)|emit_stream))",
                "blocks": r"^(scan_blocks)?$", "blocks_no_tma": r"^(?!.*(filter\(tma\)|emit_stream))"}
VARIANTS = {k: v[0] for k, v in VARIANT_DEFS.items()}


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("gpu")
    rng = np.random.default_rng(7)
    tables = {}
    tables["t"] = make_table(d, "t", 50_000, 64, 5, seed=2)                               # 156 segments: lexicographic order matters
    tables["neg"] = make_table(d, "neg", 20_000, 32, 10, seed=3, id_mode="random")        # full int8 / int32 ranges
    tables["p"] = make_table(d, "p", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    tables["pr"] = make_table(d, "pr", 5_000, 128, 4, seed=5, id_codec="PFOR_INT", id_mode="random")  # unsorted -> b=32 raw mini-blocks
    tables["ps"] = make_table(d, "ps", 9_000, 1000, 2, seed=6, id_codec="PFOR_INT")       # block size not a multiple of 32: var-byte tails
    n = 12_345
    extra = [("name:DENSE_STRING:size=5", np.array([b"alice", b"bobby", b"carol", b"dave_", b"erin#"], "S5")[rng.integers(0, 5, n)]),
             ("code:DENSE_STRING:size=1", np.array([b"x", b"y", b"z"], "S1")[rng.integers(0, 3, n)]),
             ("zip:DENSE_STRING:size=4", np.array([b"1234", b"9876", b"0000"], "S4")[rng.integers(0, 3, n)]),
             ("score:DENSE_INT", rng.integers(-1000, 1000, n).astype(np.int32))]
    tables["wide"] = make_table(d, "wide", n, 100, 7, seed=8, extra_cols=extra)
    tables["test_100"] = make_table(d, "test_100", 100, 1024, 1000, seed=2)               # README config 1
    tables["one"] = make_table(d, "one", 1, 8, 2, seed=2)
    tables["tile"] = make_table(d, "tile", 8192, 1024, 1000, seed=2)                      # exactly two dense tiles
    tables["tile1"] = make_table(d, "tile1", 4097, 1024, 1000, seed=2)
    orc = O.Oracle(d)
    sms = {k: SegmentManager(d, flags=f) for k, f in VARIANTS.items()}
    yield d, tables, orc, sms
    os.environ.pop("IMM3_PATH", None)
    for s in sms.values():
        s.close()
    orc.close()


def set_path(variant):
    path = VARIANT_DEFS.get(variant.split("/")[0], (0, ""))[1]
    if path:
        os.environ["IMM3_PATH"] = path
    else:
        os.environ.pop("IMM3_PATH", None)


def check(orc, sm, table, select, proj, limit=0, variant="", route=None):
    """Rows, values and order against the oracle; `route`: a regex the query's kernel route (Result.route) must match."""
    set_path(variant)
    exp = orc.query(table, oracle_preds(select), proj, limit=limit)
    with Engine(sm).execute(Query(table, select, Project(proj, limit))) as got:
        for want in (route, ROUTE_CHECKS.get(variant.split("/")[0])):
            assert want is None or re.search(want, got.route), (variant, table, select, proj, limit, got.route, want)
        assert got.nrows == exp.nrows, (variant, table, select, proj, limit, got.nrows, exp.nrows)
        for c in range(len(proj)):
            a, b = got.column(c), exp.columns[c]
            if not np.array_equal(a, b):
                bad = int(np.flatnonzero(a != b)[0])
                raise AssertionError(f"{variant} {table} {select} col {proj[c]} limit {limit}: first mismatch at row {bad}: got {a[bad]!r} want {b[bad]!r}")
        return got.nrows


QUERIES_T = [
    (conj(Select("age", GT(18)), Select("age", LT(30))), ["id", "age"]),                                   # C2
    (conj(Select("state", Match(["CA"])), Select("age", GT(18)), Select("age", LT(30))), ["id", "state", "age"]),  # C3
    (conj(Select("age", GT(0)), Select("state", Match(["DC", "CT"]))), ["age", "state"]),                  # Engine.scala:39-46
    (Select("age", GT(30)), ["age", "state", "id"]),                                                       # Engine.scala:48-52
    (conj(Select("id", GT(30_000)), Select("id", LT(31_500))), ["id"]),                                    # C4 shape (dense twin)
    (Select("age", EQ(7)), ["id"]),
    (Select("id", EQ(5 + 3 * 777)), ["id", "age", "state"]),
    (NoSelect, ["id", "state", "age"]),
    (NoSelect, ["age"]),
    (Select("age", LT(1)), ["id"]),
    (Or(Select("age", GT(50)), Select("age", LT(10))), ["id"]),                                            # OR == AND: empty
    (Select("state", Match(["CAL"])), ["id"]),                                                             # wrong length: empty
    (Select("age", GT(98)), ["state", "state", "id", "age", "id"]),                                        # duplicates, select-list order
    (conj(Select("age", GT(10)), Select("id", LT(100_000)), Select("state", Match(STATES[:25])), Select("age", LT(90))), ["state", "id"]),
]


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_dense_table_queries(world, variant):
    d, tables, orc, sms = world
    total = 0
    for sel, proj in QUERIES_T:
        total += check(orc, sms[variant], "t", sel, proj, 0, variant)
    assert total > 50_000


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_limit_is_an_exact_cut_in_canonical_order(world, variant):
    d, tables, orc, sms = world
    sel = conj(Select("age", GT(18)), Select("age", LT(30)))
    full = check(orc, sms[variant], "t", sel, ["id", "age"], 0, variant)
    for limit in (1, 2, 10, 63, 64, 65, 4095, 4096, 4097, full - 1, full, full + 1, 10**9):
        check(orc, sms[variant], "t", sel, ["id", "age"], limit, variant)
    for limit in (1, 10, 49_999, 50_000, 50_001):
        check(orc, sms[variant], "t", NoSelect, ["id"], limit, variant)
    check(orc, sms[variant], "t", Select("age", EQ(127)), ["id"], 5, variant)  # nothing matches, LIMIT never reached


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_narrowing_and_signed_ranges(world, variant):
    d, tables, orc, sms = world
    for sel in [Select("age", GT(200)), Select("age", EQ(300)), Select("age", LT(1e10)), Select("age", GT(-129)), Select("age", LT(-128)),
                Select("age", GT(126)), Select("age", LT(-127)), Select("age", EQ(-128)), Select("age", EQ(127)),
                Select("id", GT(3e9)), Select("id", LT(3e9)), Select("id", LT(-3e9)), Select("id", GT(-3e9)), Select("id", EQ(-2**31)),
                Select("id", EQ(2**31 - 1)), Select("id", GT(2**31 - 2)), Select("id", LT(-2**31 + 1)), Select("id", EQ(float("nan"))),
                conj(Select("id", GT(-1000.9)), Select("id", LT(1000.9))), conj(Select("id", GT(-3e9)), Select("age", LT(-5))),
                conj(Select("age", GT(-100)), Select("age", LT(100)), Select("age", GT(-50)), Select("age", LT(50)))]:
        check(orc, sms[variant], "neg", sel, ["id", "age"], 0, variant)


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_string_widths_and_extra_columns(world, variant):
    d, tables, orc, sms = world
    for sel, proj in [
        (Select("name", Match(["carol"])), ["id", "name"]),
        (Select("name", Match(["alice", "erin#", "nobody"])), ["name", "code", "zip", "score"]),
        (Select("code", Match(["y"])), ["code", "id"]),
        (Select("zip", Match(["9876", "0000"])), ["zip", "age"]),
        (conj(Select("zip", Match(["1234"])), Select("code", Match(["x", "z"])), Select("score", GT(0)), Select("age", LT(50)), Select("state", Match(["TX", "NY", "CA"]))), ["id", "name", "score"]),
        (conj(Select("score", GT(-10)), Select("score", LT(10))), ["score", "name"]),
        (NoSelect, ["name", "code", "zip", "score", "id", "state", "age"]),
    ]:
        check(orc, sms[variant], "wide", sel, proj, 0, variant)
        check(orc, sms[variant], "wide", sel, proj, 17, variant)


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_edge_sizes(world, variant):
    d, tables, orc, sms = world
    sel = conj(Select("age", GT(18)), Select("age", LT(30)))
    for table in ("test_100", "one", "tile", "tile1"):
        for limit in (0, 1, 10):
            check(orc, sms[variant], table, sel, ["id", "age"], limit, variant)
            check(orc, sms[variant], table, NoSelect, ["id", "state", "age"], limit, variant)
    check(orc, sms[variant], "t", NoSelect, [], 0, variant)  # empty select list: only the row count


@pytest.mark.parametrize("filter_stages,emit_stages", [(2, 2), (2, 3), (2, 4), (3, 2), (3, 3), (3, 4), (6, 2), (6, 3), (6, 4)])
def test_dense_tile_shapes(world, filter_stages, emit_stages, monkeypatch):
    """Every TMA ring depth of the dense filter kernel (IMM3_FILTER_STAGES, 8192-row stages) and of the streaming emit kernel
    (IMM3_EMIT_STAGES) gives the same rows: multi-round selection vectors (NoSelect fills a tile with matches), partial last
    tiles, LIMIT cuts inside and across tiles; the direct-load filter kernel (OPEN_NO_TMA, "multi_direct") alongside."""
    d, tables, orc, sms = world
    monkeypatch.setenv("IMM3_FILTER_STAGES", str(filter_stages))
    monkeypatch.setenv("IMM3_EMIT_STAGES", str(emit_stages))
    # the filter kernel's ring as asked (every filter below fits 6 stages of 8192 rows in 200 KB); a streaming emit kernel, when
    # the result density makes it run, with its ring as asked
    route = rf"^(?!.*emit_stream/s=(?!{emit_stages}(;|$))).*(^|;)filter\(tma\)/s={filter_stages}(;|$)"
    for variant in ("multi", "multi_direct"):
        for sel, proj in QUERIES_T[:5] + [(NoSelect, ["id", "state", "age"])]:
            for limit in (0, 10, 8191, 8193, 20_000):
                check(orc, sms[variant], "t", sel, proj, limit, f"{variant}/F{filter_stages}/E{emit_stages}",
                      route=route if variant == "multi" and sel is not NoSelect else None)
        check(orc, sms[variant], "wide", Select("name", Match(["carol"])), ["id", "name", "zip"], 0, f"{variant}/F{filter_stages}")
        set_path(variant)
        got, nsel = Engine(sms[variant]).filter_bitmap("t", Select("age", LT(50)))
        want, wsel = orc.filter_bitmap("t", oracle_preds(Select("age", LT(50))))
        assert nsel == wsel and np.array_equal(got, want)
    monkeypatch.setenv("IMM3_EMIT", "stream")  # the streaming emit kernel takes every result
    for limit in (0, 8193):
        check(orc, sms["multi"], "t", QUERIES_T[0][0], QUERIES_T[0][1], limit, "multi/stream", route=rf";emit_stream/s={emit_stages}$")


def test_readme_cli_query_and_row_format(world):
    d, tables, orc, sms = world
    sql = "select id, age from test_100 where (age > 18 and age < 30) limit 10"      # README.md:6
    exp = orc.query("test_100", [("age", O.OP_GT, 18), ("age", O.OP_LT, 30)], ["id", "age"], limit=10, fmt_rows=10)
    assert exp.ref_throw == 0  # inside the reference's own well-defined domain
    for variant, sm in sms.items():
        with Engine(sm).execute_sql(sql) as got:
            assert [got.format_row(i) for i in range(got.nrows)] == exp.format_rows(), variant
            assert [str(r) for r in got] == exp.format_rows()
    with Engine(sms["auto"]).execute_sql("select state, id from t where (state = 'CA' and age > 18 and age < 30) limit 3") as got:
        e2 = orc.query("t", [("state", O.OP_MATCH, ["CA"]), ("age", O.OP_GT, 18), ("age", O.OP_LT, 30)], ["state", "id"], limit=3, fmt_rows=3)
        assert [got.format_row(i) for i in range(got.nrows)] == e2.format_rows()


@pytest.mark.parametrize("table", ["p", "pr", "ps"])
def test_sorted_int_codec_tables(world, table):
    d, tables, orc, sms = world
    sm = sms["auto"]  # PFOR columns always take the block-mode kernel
    ids = tables[table]["id"]
    lo, hi = int(np.percentile(ids, 40)), int(np.percentile(ids, 60))
    for sel, proj in [
        (conj(Select("id", GT(lo)), Select("id", LT(hi))), ["id"]),                                        # C4
        (conj(Select("id", GT(lo)), Select("id", LT(hi)), Select("age", GT(18)), Select("age", LT(30))), ["id", "age", "state"]),
        (NoSelect, ["id"]),
        (NoSelect, ["id", "age", "state"]),
        (Select("age", GT(90)), ["id"]),                                                                   # PFOR column only projected
        (Select("state", Match(["CA", "NY"])), ["state", "id"]),
        (Select("id", EQ(int(ids[len(ids) // 2]))), ["id", "age"]),
        (Select("id", GT(3e9)), ["id"]),
    ]:
        for limit in (0, 1, 100, 1025):
            check(orc, sm, table, sel, proj, limit, "pfor")


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_selection_bitmap(world, variant):
    d, tables, orc, sms = world
    for table, sel in [("t", conj(Select("age", GT(18)), Select("age", LT(30)))), ("t", NoSelect), ("t", Select("state", Match(["CA"]))),
                       ("neg", Select("id", GT(0))), ("wide", Select("name", Match(["dave_"]))), ("tile1", Select("age", LT(50))),
                       ("p", Select("id", GT(1000))), ("ps", Select("age", GT(50)))]:
        set_path(variant)
        got, nsel = Engine(sms[variant]).filter_bitmap(table, sel)
        want, wsel = orc.filter_bitmap(table, oracle_preds(sel))
        assert nsel == wsel and np.array_equal(got, want), (variant, table, sel)


def test_errors_come_back_as_status_codes_not_hangs(world):
    d, tables, orc, sms = world
    eng = Engine(sms["auto"])
    for q, status in [(Query("t", Select("state", GT(1)), Project(["id"])), L.ERR_UNSUPPORTED),
                      (Query("t", Select("age", Match(["x"])), Project(["id"])), L.ERR_UNSUPPORTED),
                      (Query("t", NoSelect, Project(["nope"])), L.ERR_NOT_FOUND),
                      (Query("missing", NoSelect, Project(["id"])), L.ERR_NOT_FOUND)]:
        with pytest.raises(Imm3Error) as e:
            eng.execute(q)
        assert e.value.status == status
    check(orc, sms["auto"], "t", Select("age", GT(18)), ["id"], 10)  # the handle is still usable afterwards


@pytest.mark.parametrize("nshards", [2, 3, 8])
def test_segment_sharded_execution_matches_the_whole(world, nshards):
    """N handles (one per rank, here all on cuda:0) over contiguous canonical slices: concatenating
    what limit_split lets each rank emit equals the single-handle / oracle result."""
    d, tables, orc, sms = world
    shards = [SegmentManager(d, rank=r, world=nshards) for r in range(nshards)]
    try:
        for table, sel, proj in [("t", conj(Select("age", GT(18)), Select("age", LT(30))), ["id", "age"]),
                                 ("t", conj(Select("id", GT(30_000)), Select("id", LT(31_500))), ["id"]),
                                 ("p", Select("age", GT(50)), ["id", "state"])]:
            for limit in (0, 1, 10, 1000, 10**7):
                q = Query(table, sel, Project(proj, limit))
                handles = [Engine(s).begin(q) for s in shards]
                counts = [h.local_count for h in handles]
                offsets, takes = limit_split(counts, limit)
                parts = [h.fetch(t).columns() for h, t in zip(handles, takes)]
                exp = orc.query(table, oracle_preds(sel), proj, limit=limit)
                assert sum(takes) == exp.nrows, (table, limit, counts)
                for c in range(len(proj)):
                    assert np.array_equal(np.concatenate([p[c] for p in parts]), exp.columns[c]), (table, sel, limit, c)
                for h in handles:
                    h.close()
    finally:
        for s in shards:
            s.close()


def test_reupload_from_pinned_host_mirror(world):
    d, tables, orc, sms = world
    with SegmentManager(d, flags=OPEN_KEEP_HOST) as sm:
        sel = conj(Select("age", GT(18)), Select("age", LT(30)))
        check(orc, sm, "t", sel, ["id", "age"])
        assert sm.reupload("t", ["age", "id"]) == 5 * 50_000
        check(orc, sm, "t", sel, ["id", "age"])
        assert sm.reupload("t") == 7 * 50_000
        check(orc, sm, "p", Select("id", GT(100)), ["id"])
        sm.reupload("p")
        check(orc, sm, "p", Select("id", GT(100)), ["id"])


def test_async_fetch_overlaps_restaging_and_matches_sync(world):
    """imm3_result_fetch_async / imm3_result_wait: the read-back of query i runs on the copy stream while the inputs of
    query i+1 are re-staged and its kernels run; rows are identical to the synchronous fetch and to the oracle."""
    d, tables, orc, sms = world
    with SegmentManager(d, flags=OPEN_KEEP_HOST) as sm:
        eng = Engine(sm)
        sel = conj(Select("age", GT(18)), Select("age", LT(30)))
        exp = orc.query("t", oracle_preds(sel), ["id", "age"], limit=0)
        q = Query("t", sel, Project(["id", "age"]))
        prev = None
        for _ in range(4):
            sm.reupload("t", ["age", "id"])
            r = eng.begin(q)
            assert r.local_count == exp.nrows
            r.fetch_async(r.local_count)
            if prev is not None:
                prev.wait()
                assert np.array_equal(prev.column(0), exp.columns[0]) and np.array_equal(prev.column(1), exp.columns[1])
                prev.close()
            prev = r
        prev.wait().wait()  # a second wait is a no-op
        assert prev.nrows == exp.nrows and np.array_equal(prev.column(0), exp.columns[0])
        prev.close()
        r = eng.begin(q)
        r.fetch_async(10)
        r.close()  # closing with a copy in flight waits for it


def test_repeated_queries_reuse_buffers_and_epochs(world):
    d, tables, orc, sms = world
    sel = conj(Select("age", GT(18)), Select("age", LT(30)))
    for i in range(40):
        check(orc, sms["auto"], "t", sel, ["id", "age"], [0, 7, 5000][i % 3])


def test_full_size_synthetic_properties(tmp_path_factory):
    """BASELINE-shaped synthetic table (id = row index, B=1024, S=1000) at a size the oracle would need
    minutes for: checked through size-independent properties computed with numpy from the files."""
    d = tmp_path_factory.mktemp("syn")
    n = 12_000_000  # 12 segments: canonical order 0,1,10,11,2,...
    synth_write(d, "syn", n)
    order = sorted(range(12), key=lambda i: f"id_{i}.dat")
    age = np.concatenate([np.fromfile(d / "syn" / f"age_{i}.dat", np.int8) for i in order])
    ids = np.concatenate([np.fromfile(d / "syn" / f"id_{i}.dat", "<i4") for i in order])
    st = np.concatenate([np.fromfile(d / "syn" / f"state_{i}.dat", "S2") for i in order])
    set_path("auto")
    for flags in (0, OPEN_NO_TMA):
        with SegmentManager(d, flags=flags) as sm:
            eng = Engine(sm)
            m = (age > 18) & (age < 30)
            with eng.execute(Query("syn", conj(Select("age", GT(18)), Select("age", LT(30))), Project(["id", "age"]))) as r:     # C2
                assert r.nrows == int(m.sum()) and np.array_equal(r.column(0), ids[m]) and np.array_equal(r.column(1), age[m])
                assert r.algorithmic_bytes == n + r.nrows * 9 and r.kernel_launches in (2, 3)
            m3 = m & (st == b"CA")
            with eng.execute(Query("syn", conj(Select("state", Match(["CA"])), Select("age", GT(18)), Select("age", LT(30))), Project(["id", "state", "age"]))) as r:  # C3
                assert r.nrows == int(m3.sum()) and np.array_equal(r.column(0), ids[m3]) and np.all(r.column(1) == b"CA")
            lo, hi = n // 2 - n // 200, n // 2 + n // 200
            with eng.execute(Query("syn", conj(Select("id", GT(lo)), Select("id", LT(hi))), Project(["id"]))) as r:             # C4, dense twin
                mm = (ids > lo) & (ids < hi)
                assert r.nrows == hi - lo - 1 and np.array_equal(r.column(0), ids[mm])
            with eng.execute(Query("syn", Select("age", LT(50)), Project(["id"], 10))) as r:
                assert np.array_equal(r.column(0), ids[age < 50][:10])
            bm, nsel = eng.filter_bitmap("syn", Select("age", LT(50)))
            assert nsel == int((age < 50).sum())
            assert np.array_equal(np.unpackbits(bm.view(np.uint8), bitorder="little")[:n].astype(bool), age < 50)


def test_full_size_sorted_int_codec_properties(tmp_path_factory):
    d = tmp_path_factory.mktemp("synp")
    n = 12_000_000  # large enough for the prefix-first LIMIT (4 M-row prefix) to be taken at its default size
    synth_write(d, "synp", n, id_codec=L.CODEC_PFOR_INT)
    order = sorted(range(12), key=lambda i: f"id_{i}.dat")
    age = np.concatenate([np.fromfile(d / "synp" / f"age_{i}.dat", np.int8) for i in order])
    per = 1024 * 1000 + 1
    ids = np.concatenate([np.arange(i * per, min(n, (i + 1) * per), dtype=np.int32) for i in order])
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        assert sm.getTable("synp").resident_bytes < 3.4 * n   # ~0.29 B/row for the id column
        lo, hi = n // 2 - n // 200, n // 2 + n // 200
        with eng.execute(Query("synp", conj(Select("id", GT(lo)), Select("id", LT(hi))), Project(["id"]))) as r:               # C4
            mm = (ids > lo) & (ids < hi)
            assert r.nrows == hi - lo - 1 and np.array_equal(r.column(0), ids[mm])
        with eng.execute(Query("synp", conj(Select("age", EQ(7))), Project(["id", "age"]))) as r:
            assert np.array_equal(r.column(0), ids[age == 7]) and np.all(r.column(1) == 7)
        with eng.execute(Query("synp", NoSelect, Project(["id"]))) as r:
            assert np.array_equal(r.column(0), ids)
        # small LIMIT: filled by the prefix / only by the whole table (id window past the prefix) / never filled
        with eng.execute(Query("synp", Select("age", LT(10)), Project(["id", "age"], 10))) as r:
            assert r.nrows == 10 and np.array_equal(r.column(0), ids[age < 10][:10])
        with eng.execute(Query("synp", conj(Select("id", GT(lo)), Select("id", LT(hi))), Project(["id"], 1000))) as r:
            assert r.nrows == 1000 and np.array_equal(r.column(0), ids[mm][:1000])
        with eng.execute(Query("synp", conj(Select("id", GT(n - 5)), Select("age", LT(100))), Project(["id", "age"], 100))) as r:
            tail = (ids > n - 5)
            assert r.nrows == int(tail.sum()) and np.array_equal(r.column(0), ids[tail])


def test_multipass_large_limit_and_mixed_density(tmp_path_factory):
    """LIMIT > 2^20 keeps the multi-pass pipelines (dense and block mode) and must cut exactly; results whose density varies
    along the table (clustered id window = full and empty tiles, a rare age value = sparse tiles, a dense age range = streamed
    tiles) exercise every per-tile mode of the streaming emit kernel, both emit kernels and the per-shape feedback."""
    d = tmp_path_factory.mktemp("big")
    n = 2_600_000
    make_table(d, "big", n, 1024, 100, seed=12)                                             # 26 segments, dense id
    make_table(d, "bigp", n, 1024, 100, seed=12, id_codec="PFOR_INT")                     # same rows, sorted-int codec id
    os.environ.pop("IMM3_PATH", None)
    with O.Oracle(d) as orc, SegmentManager(d) as sm:
        eng = Engine(sm)
        cases = [(NoSelect, ["id", "state", "age"]),
                 (conj(Select("age", GT(10)), Select("age", LT(60))), ["age", "id"]),
                 (conj(Select("id", GT(3_000_000)), Select("id", LT(6_500_000))), ["id", "age", "state"]),
                 (Select("age", EQ(7)), ["id", "state"]),
                 (conj(Select("state", Match(["CA", "NY"])), Select("age", GT(90))), ["state", "id"])]
        for table in ("big", "bigp"):
            for sel, proj in cases:
                for limit in (0, (1 << 20) + 1, (1 << 20) + 4099, 2_500_000):
                    for _rep in range(2):  # second run: only the emit kernel remembered for this shape is launched
                        exp = orc.query(table, oracle_preds(sel), proj, limit=limit)
                        with eng.execute(Query(table, sel, Project(proj, limit))) as got:
                            assert got.nrows == exp.nrows, (table, sel, limit, got.nrows, exp.nrows)
                            for c in range(len(proj)):
                                assert np.array_equal(got.column(c), exp.columns[c]), (table, sel, proj[c], limit)


@pytest.mark.gpu
@pytest.mark.parametrize("block_rows", [1024, 256, 32])
def test_gpu_sorted_int_encoder_is_bit_exact(block_rows):
    """imm3_pfor_encode_blocks_gpu == the ORACLE's PFORCodecInt.encode (and the product's host encoder) block by block: sorted
    ids, equal values (width 0), wide and negative deltas (width 32, raw mini-blocks), every tail length, one short block."""
    from immutable3_b200.loader import pfor_encode, pfor_encode_blocks_gpu
    rng = np.random.default_rng(7 + block_rows)
    cols = {
        "row index": np.arange(10 * block_rows + 17, dtype=np.int64),
        "steps": np.cumsum(rng.integers(0, 1000, 7 * block_rows + 5)),
        "constant": np.full(3 * block_rows, 12345, dtype=np.int64),
        "mixed widths": np.cumsum(np.where(rng.random(9 * block_rows + 31) < 0.02, rng.integers(0, 1 << 20, 9 * block_rows + 31), rng.integers(0, 4, 9 * block_rows + 31))),
        "unsorted": rng.integers(-2**31, 2**31 - 1, 5 * block_rows + 1),
        "short": np.arange(7, dtype=np.int64) * 300,
        "one": np.array([300], dtype=np.int64),
        "worksheet": np.array([1, 2, 3, 4, 5, 100, 120, 123, 150, 121, 122, 123, 125, 1000, 1100], dtype=np.int64),  # exploration/compression.sc:6
    }
    for tail in range(0, 33, 5):
        cols[f"tail {tail}"] = np.cumsum(rng.integers(0, 70000, 2 * block_rows + tail))
    for name, v in cols.items():
        v = v.astype(np.int64).astype(np.int32) if v.dtype != np.int32 else v
        got, off = pfor_encode_blocks_gpu(v, block_rows)
        exp = [O.pfor_encode(v[i:i + block_rows]) for i in range(0, len(v), block_rows)]   # the checker, directly
        assert list(np.diff(off)) == [len(e) for e in exp], name
        assert got == b"".join(exp), name
        assert exp == [pfor_encode(v[i:i + block_rows]) for i in range(0, len(v), block_rows)], name


def test_several_sorted_int_codec_columns(tmp_path_factory):
    """Three encoded columns in one table: predicates on one or two of them (one decode per predicate column in the
    filter kernel), all of them in the select list (several decoded columns side by side in the emit kernel), a select
    list of more than four columns (the column-by-column emit path), with and without LIMIT."""
    d = tmp_path_factory.mktemp("multi_pfor")
    n = 70_000
    rng = np.random.default_rng(21)
    ts = np.cumsum(rng.integers(0, 50, n)).astype(np.int32)
    k2 = np.cumsum(rng.choice([0, 1, 70000], size=n, p=[0.5, 0.49, 0.01])).astype(np.int32)
    make_table(d, "mp", n, 1024, 20, seed=3, id_codec="PFOR_INT", extra_cols=[("ts:PFOR_INT", ts), ("k2:PFOR_INT", k2), ("v:DENSE_INT", (ts // 7).astype(np.int32))])
    os.environ.pop("IMM3_PATH", None)
    with O.Oracle(d) as orc, SegmentManager(d) as sm:
        eng = Engine(sm)
        cases = [(conj(Select("ts", GT(int(ts[n // 3]))), Select("ts", LT(int(ts[n // 2])))), ["id", "ts", "k2"]),
                 (conj(Select("ts", GT(int(ts[n // 4]))), Select("k2", LT(int(k2[3 * n // 4]))), Select("age", LT(40))), ["k2", "age", "ts"]),
                 (Select("age", EQ(7)), ["ts", "id", "k2", "v"]),
                 (conj(Select("id", GT(30_000)), Select("v", LT(int(ts[n // 2]) // 7))), ["id", "state", "age", "ts", "k2", "v"]),
                 (NoSelect, ["k2", "ts"])]
        for sel, proj in cases:
            for limit in (0, 10, 3000):
                exp = orc.query("mp", oracle_preds(sel), proj, limit=limit)
                with eng.execute(Query("mp", sel, Project(proj, limit))) as got:
                    assert got.nrows == exp.nrows, (sel, limit, got.nrows, exp.nrows)
                    for c in range(len(proj)):
                        assert np.array_equal(got.column(c), exp.columns[c]), (sel, proj[c], limit)


def test_small_limit_runs_prefix_first(tmp_path_factory, monkeypatch):
    """Small LIMIT (here on a table with a sorted-int-codec column and on its dense twin): the pipeline first covers a prefix of the blocks and only
    scans the whole table when the prefix does not fill the LIMIT.  Rows found early, late (id window at the end), never,
    and a LIMIT that the prefix fills only partly must all give the oracle's exact cut."""
    d = tmp_path_factory.mktemp("pfx")
    n = 300_000
    make_table(d, "pp", n, 1024, 40, seed=5, id_codec="PFOR_INT")
    make_table(d, "pd", n, 1024, 40, seed=5)  # dense twin: the same policy on the dense multi-pass pipeline
    monkeypatch.setenv("IMM3_PREFIX_ROWS", "8192")
    os.environ.pop("IMM3_PATH", None)
    with O.Oracle(d) as orc, SegmentManager(d) as sm:
        eng = Engine(sm)
        cases = [(Select("age", LT(10)), ["id", "age"]),                                             # early, dense filter (row-space path)
                 (conj(Select("id", GT(250_000)), Select("id", LT(260_000))), ["id", "state"]),       # late, filter on the encoded column
                 (conj(Select("id", GT(4_000)), Select("age", EQ(7))), ["age", "id"]),                # straddles the prefix
                 (conj(Select("state", Match(["CA"])), Select("age", EQ(3))), ["id", "state", "age"]),  # rare rows
                 (Select("age", EQ(127)), ["id"]),                                                     # no rows at all
                 (NoSelect, ["id"])]
        for table in ("pp", "pd"):
            for sel, proj in cases:
                for limit in (1, 10, 100, 5000):
                    exp = orc.query(table, oracle_preds(sel), proj, limit=limit)
                    with eng.execute(Query(table, sel, Project(proj, limit))) as got:
                        assert got.nrows == exp.nrows, (table, sel, limit, got.nrows, exp.nrows)
                        for c in range(len(proj)):
                            assert np.array_equal(got.column(c), exp.columns[c]), (table, sel, proj[c], limit)


@pytest.mark.parametrize("seed", list(range(10)) + [118])  # 118: LIMIT == number of matches on 1500 small blocks (look-back abort race)
def test_random_tables_and_queries(tmp_path_factory, seed):
    """Randomised end-to-end parity: table shape (rows, block size, segment size, id codec and order), predicate set, select
    list and LIMIT are drawn from a seeded generator; the default kernel choice and the forced single-pass kernels must both
    reproduce the oracle's rows, values and order."""
    seed += int(os.environ.get("IMM3_TEST_SEED_BASE", "0"))  # (stress runs: other seeds without editing the file)
    rng = np.random.default_rng(1000 + seed)
    d = tmp_path_factory.mktemp(f"rnd{seed}")
    nrows = int(rng.choice([1, 31, 1000, 8191, 8193, 40_000, 150_000]))
    block = int(rng.choice([8, 32, 100, 1000, 1024, 4096]))
    segment = int(rng.integers(1, 40))
    codec = "PFOR_INT" if rng.random() < 0.4 else "DENSE_INT"
    mode = str(rng.choice(["sorted", "steps", "random"]))
    cols = make_table(d, "r", nrows, block, segment, seed=int(rng.integers(0, 100)), id_codec=codec, id_mode=mode)
    ids, ages = cols["id"].astype(np.int64), cols["age"].astype(np.int64)

    def random_select():
        leaves = []
        for _ in range(int(rng.integers(0, 4))):
            kind = rng.integers(0, 5)
            if kind == 0:
                leaves.append(Select("age", GT(float(rng.integers(-140, 140)))))
            elif kind == 1:
                leaves.append(Select("age", LT(float(rng.integers(-140, 140)) + 0.5)))
            elif kind == 2:
                q = float(np.quantile(ids, rng.random()))
                leaves.append(Select("id", GT(q)) if rng.random() < 0.5 else Select("id", LT(q)))
            elif kind == 3:
                leaves.append(Select("state", Match([str(s) for s in rng.choice(STATES, size=int(rng.integers(1, 6)))])))
            else:
                leaves.append(Select("age", EQ(float(ages[int(rng.integers(0, nrows))]))))
        return conj(*leaves)

    with O.Oracle(d) as orc:
        for path in ("", "fused"):
            if path:
                os.environ["IMM3_PATH"] = path
            else:
                os.environ.pop("IMM3_PATH", None)
            with SegmentManager(d) as sm:
                eng = Engine(sm)
                for _q in range(12):
                    sel = random_select()
                    proj = [str(c) for c in rng.choice(["id", "state", "age"], size=int(rng.integers(0, 5)))]
                    limit = int(rng.choice([0, 0, 1, 7, 1000, nrows, nrows + 5]))
                    exp = orc.query("r", oracle_preds(sel), proj, limit=limit)
                    with eng.execute(Query("r", sel, Project(proj, limit))) as got:
                        assert got.nrows == exp.nrows, (seed, path, sel, proj, limit, got.nrows, exp.nrows)
                        for c in range(len(proj)):
                            assert np.array_equal(got.column(c), exp.columns[c]), (seed, path, sel, proj[c], limit)
    os.environ.pop("IMM3_PATH", None)


def _shape_ids(shape, n, rng):
    """int32 id columns that walk the sorted-integer codec's block shapes (widths, raw mini-blocks, wrap-around)."""
    kind, arg = shape
    if kind == "const":      # constant delta: every mini-block has the same width
        start, d = arg
        v = start + d * np.arange(n, dtype=np.int64)
    elif kind == "bits":     # random deltas below 2^b (cumulative sum wraps mod 2^32 for large b)
        v = np.cumsum(rng.integers(0, 1 << arg, size=n, dtype=np.int64)) + int(rng.integers(-2**31, 2**31))
    elif kind == "mixed":    # mostly width 1-2, a few wide jumps, a few repeats, a run of unsorted values (raw mini-blocks)
        d = rng.choice([0, 1, 1, 1, 2, 3, 1 << arg], size=n, p=[0.1, 0.3, 0.2, 0.2, 0.1, 0.09, 0.01]).astype(np.int64)
        v = np.cumsum(d) - 2**31 + 17
        if n > 300:
            a = int(rng.integers(0, n - 200))
            v[a:a + 150] = rng.integers(-2**31, 2**31, size=150)
    else:                    # unsorted: every mini-block raw
        v = rng.integers(-2**31, 2**31, size=n, dtype=np.int64)
    return ((v + 2**31) % 2**32 - 2**31).astype(np.int32)


SHAPES = [("const", (0, 0)), ("const", (5, 1)), ("const", (-2**31, 2)), ("const", (7, 3)), ("const", (100, 15)), ("const", (0, 16)),
          ("const", (-1000, 255)), ("const", (3, 256)), ("const", (2**31 - 70_000 * 4 - 2, 4)), ("const", (0, 65535)), ("const", (-2**31, 30000)),
          ("bits", 1), ("bits", 2), ("bits", 3), ("bits", 4), ("bits", 7), ("bits", 8), ("bits", 9), ("bits", 13), ("bits", 16), ("bits", 20),
          ("bits", 26), ("bits", 27), ("bits", 30), ("mixed", 10), ("mixed", 24), ("mixed", 29), ("random", 0)]


@pytest.mark.parametrize("prune", [True, False])
@pytest.mark.parametrize("block", [1024, 1000, 640, 256, 160, 128, 32])
def test_sorted_int_codec_range_predicates_over_block_shapes(tmp_path_factory, block, prune, monkeypatch):
    """The filter kernel of the sorted-integer codec classifies whole mini-blocks from their packed words (k_blocks_filter.cuh):
    every width class, raw mini-blocks, wrap-around past 2^31 / 2^32, window edges on and next to mini-block boundaries."""
    from immutable3_b200.loader import SegmentWriter

    if not prune:
        monkeypatch.setenv("IMM3_NO_PRUNE", "1")  # (default: whole blocks are decided from their min / max first, k_blocks_prune.cuh)
    d = tmp_path_factory.mktemp(f"shapes{block}")
    rng = np.random.default_rng(block)
    n = 70_000 if block >= 1000 else 9_000
    cols = {}
    for i, shape in enumerate(SHAPES):
        ids = _shape_ids(shape, n, rng)
        ages = rng.integers(0, 100, size=n).astype(np.int8)
        with SegmentWriter(d, f"s{i}", ["id:PFOR_INT", "age:DENSE_TINYINT"], block, 11) as w:
            w.append(ids, ages)
        cols[f"s{i}"] = ids
    os.environ.pop("IMM3_PATH", None)
    with O.Oracle(d) as orc, SegmentManager(d) as sm:
        eng = Engine(sm)
        for name, ids in cols.items():
            picks = [int(ids[int(j)]) for j in rng.integers(0, n, size=6)] + [int(ids[0]), int(ids[31]), int(ids[32]), int(ids[-1]), int(ids.min()), int(ids.max())]
            sels = []
            for a in picks[:6]:
                b = picks[int(rng.integers(0, len(picks)))]
                lo, hi = min(a, b), max(a, b)
                sels += [conj(Select("id", GT(lo)), Select("id", LT(hi))), conj(Select("id", GT(lo - 1)), Select("id", LT(hi + 1)))]
            sels += [Select("id", EQ(picks[1])), Select("id", GT(picks[8])), Select("id", LT(picks[7])), Select("id", GT(-3e9)), Select("id", LT(-3e9)),
                     conj(Select("id", GT(picks[2])), Select("age", LT(50))), Select("id", EQ(int(ids.min()))), Select("id", GT(int(ids.max()) - 1))]
            for sel in sels:
                for limit in (0, 33):
                    exp = orc.query(name, oracle_preds(sel), ["id"], limit=limit)
                    with eng.execute(Query(name, sel, Project(["id"], limit))) as got:
                        assert got.nrows == exp.nrows, (name, SHAPES[int(name[1:])], sel, limit, got.nrows, exp.nrows)
                        assert np.array_equal(got.column(0), exp.columns[0]), (name, SHAPES[int(name[1:])], sel, limit)


def test_offset_scan_kernel_on_large_and_small_tables(tmp_path_factory, world, monkeypatch):
    """Tables with more than 16 K tiles hand the tile-count scan to offset_scan_kernel (one CTA per 4096 counts, chained sums);
    IMM3_SCAN=kernel forces it everywhere: multi-chunk dense and block tables, the small fixtures, LIMIT cuts."""
    monkeypatch.setenv("IMM3_SCAN", "kernel")
    os.environ.pop("IMM3_PATH", None)
    d, tables, orc, sms = world
    for table, sel, proj in [("t", conj(Select("age", GT(18)), Select("age", LT(30))), ["id", "age"]), ("t", NoSelect, ["id"]),
                             ("p", conj(Select("id", GT(2000)), Select("id", LT(900000))), ["id", "age"]), ("p", Select("age", LT(10)), ["id"]),
                             ("wide", Select("name", Match(["carol"])), ["id", "name", "zip"]), ("one", NoSelect, ["id"])]:
        for limit in (0, 1, 100, 5000):
            check(orc, sms["auto"], table, sel, proj, limit, "auto")
    # 40 M rows: 4883 dense tiles -> 2 chunks; checked with numpy from the files
    d2 = tmp_path_factory.mktemp("scan")
    n = 40_000_000
    synth_write(d2, "syn", n)
    order = sorted(range(40), key=lambda i: f"id_{i}.dat")
    age = np.concatenate([np.fromfile(d2 / "syn" / f"age_{i}.dat", np.int8) for i in order])
    ids = np.concatenate([np.fromfile(d2 / "syn" / f"id_{i}.dat", "<i4") for i in order])
    # a block table with small blocks: 3 M rows in blocks of 32 -> 11.7 K tiles of 8 blocks -> 3 chunks
    rng = np.random.default_rng(5)
    nb = 3_000_000
    bid = np.cumsum(rng.integers(0, 4, size=nb)).astype(np.int32)
    bage = rng.integers(0, 100, size=nb).astype(np.int8)
    from immutable3_b200.loader import SegmentWriter
    with SegmentWriter(d2, "b32", ["id:PFOR_INT", "age:DENSE_TINYINT"], 32, 1000) as w:
        w.append(bid, bage)
    border = np.concatenate([np.arange(i * 32001, min(nb, (i + 1) * 32001)) for i in sorted(range((nb + 32000) // 32001), key=lambda i: f"id_{i}.dat")])
    with SegmentManager(d2) as sm:
        eng = Engine(sm)
        for lim in (0, 1000, 3_000_000):
            m = (age > 18) & (age < 30)
            with eng.execute(Query("syn", conj(Select("age", GT(18)), Select("age", LT(30))), Project(["id", "age"], lim))) as r:
                want = ids[m][:lim] if lim else ids[m]
                assert r.nrows == len(want) and np.array_equal(r.column(0), want) and r.kernel_launches >= 3
            lo, hi = int(bid[nb // 3]), int(bid[2 * nb // 3])
            cb, ca = bid[border], bage[border]
            mb = (cb > lo) & (cb < hi)
            with eng.execute(Query("b32", conj(Select("id", GT(lo)), Select("id", LT(hi))), Project(["id", "age"], lim))) as r:
                want = cb[mb][:lim] if lim else cb[mb]
                assert r.nrows == len(want) and np.array_equal(r.column(0), want) and np.array_equal(r.column(1), (ca[mb][:lim] if lim else ca[mb]))
            with eng.execute(Query("b32", Select("age", LT(3)), Project(["id"], lim))) as r:     # row-space filter + block emit
                want = cb[ca < 3][:lim] if lim else cb[ca < 3]
                assert r.nrows == len(want) and np.array_equal(r.column(0), want)


@pytest.mark.parametrize("scanemit", [True, False])
def test_dense_sorted_ids_at_every_start_width(tmp_path_factory, scanemit, monkeypatch):
    """The lane-per-block filter kernel (k_blocks_lane.cuh) reads the wide first mini-block of a dense sorted block with its width
    B folded into the code (B = 17 .. 31, LDS.128 chunks when blocks are 0 mod 4 words) and walks it generically below that;
    blocks_scan_emit_kernel decodes the same shape straight from global memory.  Ids that start just below a power of two put
    both widths into one tile; several segments put 1-row tail blocks at every lane; block size 72 words = the 8-way bank case.
    Checked against numpy and - IMM3_NO_SCANEMIT=1 - through the general scan + emit kernels as well."""
    from immutable3_b200.loader import SegmentWriter

    if not scanemit:
        monkeypatch.setenv("IMM3_NO_SCANEMIT", "1")
    os.environ.pop("IMM3_PATH", None)
    d = tmp_path_factory.mktemp("widths")
    n = 140_001
    rng = np.random.default_rng(3)
    tables = {}
    for i, base in enumerate([0, (1 << 17) - 3000, (1 << 22) - 5000, (1 << 26) - 9000, (1 << 29) - 40_000, (1 << 30) - 70_000, (1 << 31) - 140_001]):
        ids = (np.arange(n, dtype=np.int64) + base).astype(np.int32)
        with SegmentWriter(d, f"w{i}", ["id:PFOR_INT"], 1024, 14 + i) as w:  # 14 .. 20 blocks per segment (<= 10 segments: file-name order = id order): tail blocks at many lanes
            w.append(ids)
        tables[f"w{i}"] = ids
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        for name, ids in tables.items():
            b = int(ids[0])
            windows = [(b + 1000, b + 90_000), (b + 1023, b + 1025), (b + 1024 * 31, b + 1024 * 33 + 1), (b - 5, b + 5), (b + n - 3, b + n + 5),
                       (b + 33_333, b + 33_334), (b - 10, b + n + 10), (b + 70_000, b + 70_000)]
            windows += [tuple(sorted(int(x) for x in rng.integers(b, b + n, size=2))) for _ in range(4)]
            for lo, hi in windows:
                hi = min(hi, (1 << 31) - 1)  # (constants stay inside the Int range: the narrowing rules have their own test)
                sel = conj(Select("id", GT(lo)), Select("id", LT(hi)))
                want = ids[(ids.astype(np.int64) > lo) & (ids.astype(np.int64) < hi)]
                for limit in (0, 10, 2000, 70_001):
                    with eng.execute(Query(name, sel, Project(["id"], limit))) as got:
                        exp = want if limit == 0 else want[:limit]
                        assert got.nrows == len(exp), (name, lo, hi, limit, got.nrows, len(exp))
                        assert np.array_equal(got.column(0), exp), (name, lo, hi, limit)


@pytest.mark.parametrize("groupemit", [True, False])
def test_scan_emit_kernel_over_several_scan_chunks(tmp_path_factory, groupemit, monkeypatch):
    """blocks_scan_emit_kernel with more than one scan chunk (3 M rows in blocks of 32 rows: 11.7 K tiles of 8 blocks, 3 chunks of
    4096), sparse and dense windows, LIMIT cuts inside blocks - gaps of 0 .. 3 between ids give mini-blocks of widths 0 .. 2.
    By default blocks_group_emit_kernel serves these queries (92 groups of 1024 blocks); IMM3_NO_GROUPEMIT=1 keeps the scan-emit kernel."""
    from immutable3_b200.loader import SegmentWriter

    if not groupemit:
        monkeypatch.setenv("IMM3_NO_GROUPEMIT", "1")
    os.environ.pop("IMM3_PATH", None)
    d = tmp_path_factory.mktemp("chunks")
    rng = np.random.default_rng(11)
    n = 3_000_000
    ids = np.cumsum(rng.integers(0, 4, size=n)).astype(np.int32)
    with SegmentWriter(d, "c", ["id:PFOR_INT"], 32, 20_000) as w:
        w.append(ids)
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        top = int(ids[-1])
        for lo, hi in [(-1, top + 1), (top // 3, top // 3 + 50), (top // 2, top // 2 + 400_000), (top - 10, top + 10), (5, 6)]:
            sel = conj(Select("id", GT(lo)), Select("id", LT(hi)))
            want = ids[(ids > lo) & (ids < hi)]
            for limit in (0, 1, 33, 5000, 1_000_001):
                with eng.execute(Query("c", sel, Project(["id"], limit))) as got:
                    exp = want if limit == 0 else want[:limit]
                    assert got.nrows == len(exp), (lo, hi, limit, got.nrows, len(exp))
                    assert np.array_equal(got.column(0), exp), (lo, hi, limit)


@pytest.mark.parametrize("prune", [True, False])
def test_group_emit_kernel_many_blocks_per_cta(tmp_path_factory, prune, monkeypatch):
    """blocks_group_emit_kernel (k_blocks_groupemit.cuh): 8 M rows in blocks of 32 rows = 250 K blocks in 245 groups - a CTA's share
    of a group exceeds its 256-entry queue (several rounds), CTA ranges span group boundaries, LIMIT cuts fall inside blocks and
    on block / group boundaries; a second table whose every block is partially selected (bitmap words for every block); both
    with and without block pruning (the prune kernel adds the group sums of the blocks it decides)."""
    from immutable3_b200.loader import SegmentWriter

    if not prune:
        monkeypatch.setenv("IMM3_NO_PRUNE", "1")
    os.environ.pop("IMM3_PATH", None)
    d = tmp_path_factory.mktemp("groups")
    rng = np.random.default_rng(23)
    n = 8_000_000
    ids = np.cumsum(rng.integers(0, 3, size=n)).astype(np.int32)
    with SegmentWriter(d, "g", ["id:PFOR_INT"], 32, 50_000) as w:
        w.append(ids)
    m = 600_000
    saw = ((np.arange(m) % 64) * 3 + (np.arange(m) // 64) % 2).astype(np.int32)  # every 32-row block holds half a ramp
    with SegmentWriter(d, "saw", ["id:PFOR_INT"], 32, 3_000) as w:
        w.append(saw)
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        top = int(ids[-1])
        for lo, hi in [(-1, top + 1), (top // 4, 3 * (top // 4)), (top // 2, top // 2 + 70), (int(ids[32 * 1024 * 7]) - 1, int(ids[32 * 1024 * 9]))]:
            sel = conj(Select("id", GT(lo)), Select("id", LT(hi)))
            want = ids[(ids > lo) & (ids < hi)]
            for limit in (0, 1, 32 * 1024, 32 * 1024 + 5, 4_000_000):
                with eng.execute(Query("g", sel, Project(["id"], limit))) as got:
                    exp = want if limit == 0 else want[:limit]
                    assert got.nrows == len(exp), (lo, hi, limit, got.nrows, len(exp))
                    assert np.array_equal(got.column(0), exp), (lo, hi, limit)
        for lo, hi in [(20, 170), (-1, 50), (95, 97), (190, 1000)]:
            sel = conj(Select("id", GT(lo)), Select("id", LT(hi)))
            want = saw[(saw > lo) & (saw < hi)]
            for limit in (0, 77, 100_000):
                with eng.execute(Query("saw", sel, Project(["id"], limit))) as got:
                    exp = want if limit == 0 else want[:limit]
                    assert got.nrows == len(exp), ("saw", lo, hi, limit, got.nrows, len(exp))
                    assert np.array_equal(got.column(0), exp), ("saw", lo, hi, limit)
    if prune:
        return
    # more than 1024 groups (34 M rows in blocks of 32): the group sums do not fit the kernel's shared-memory copy - eight per
    # thread in the CTA's scan, look-aheads from global memory
    big = np.cumsum(rng.integers(0, 2, size=34_000_000)).astype(np.int32)
    with SegmentWriter(d, "big", ["id:PFOR_INT"], 32, 200_000) as w:
        w.append(big)
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        top = int(big[-1])
        for lo, hi in [(top // 2, top // 2 + 300_000), (top - 5000, top + 1), (-1, 9), (int(big[32 * 1024 * 1030]) - 1, int(big[32 * 1024 * 1031]))]:
            sel = conj(Select("id", GT(lo)), Select("id", LT(hi)))
            want = big[(big > lo) & (big < hi)]
            for limit in (0, 100_000):
                with eng.execute(Query("big", sel, Project(["id"], limit))) as got:
                    exp = want if limit == 0 else want[:limit]
                    assert got.nrows == len(exp), ("big", lo, hi, limit, got.nrows, len(exp))
                    assert np.array_equal(got.column(0), exp), ("big", lo, hi, limit)


def test_baseline_table_at_100m_rows(tmp_path_factory):
    """BASELINE.json's test_100m (100 M rows, B = 1024, S = 1000: 98 segments, file-name order 0, 1, 10, 11, ...) and its PFOR
    twin at full size: C2, C3 and C4 against numpy evaluated on the files themselves (the oracle needs seconds per query here)."""
    d = tmp_path_factory.mktemp("syn100m")
    n = 100_000_000
    nseg = (n + 1024 * 1000) // (1024 * 1000 + 1)
    synth_write(d, "test_100m", n)
    order = sorted(range(nseg), key=lambda i: f"id_{i}.dat")
    age = np.concatenate([np.fromfile(d / "test_100m" / f"age_{i}.dat", np.int8) for i in order])
    ids = np.concatenate([np.fromfile(d / "test_100m" / f"id_{i}.dat", "<i4") for i in order])
    st = np.concatenate([np.fromfile(d / "test_100m" / f"state_{i}.dat", "S2") for i in order])
    assert len(ids) == n
    os.environ.pop("IMM3_PATH", None)
    m = (age > 18) & (age < 30)
    lo, hi = n // 2 - n // 200, n // 2 + n // 200
    mm = (ids > lo) & (ids < hi)
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        with eng.execute(Query("test_100m", conj(Select("age", GT(18)), Select("age", LT(30))), Project(["id", "age"]))) as r:     # C2
            assert r.nrows == int(m.sum()) and np.array_equal(r.column(0), ids[m]) and np.array_equal(r.column(1), age[m])
        m3 = m & (st == b"CA")
        with eng.execute(Query("test_100m", conj(Select("state", Match(["CA"])), Select("age", GT(18)), Select("age", LT(30))),
                               Project(["id", "state", "age"]))) as r:                                                              # C3
            assert r.nrows == int(m3.sum()) and np.array_equal(r.column(0), ids[m3]) and np.array_equal(r.column(2), age[m3])
        with eng.execute(Query("test_100m", conj(Select("id", GT(lo)), Select("id", LT(hi))), Project(["id"]))) as r:              # C4, dense twin
            assert np.array_equal(r.column(0), ids[mm])
    del st
    d2 = tmp_path_factory.mktemp("syn100p")
    synth_write(d2, "test_1b", n, id_codec=L.CODEC_PFOR_INT)  # (same rows, id in the sorted-integer codec: the north-star table's schema)
    with SegmentManager(d2) as sm:
        eng = Engine(sm)
        for limit in (0, 10, 123_457):
            with eng.execute(Query("test_1b", conj(Select("id", GT(lo)), Select("id", LT(hi))), Project(["id"], limit))) as r:     # C4
                exp = ids[mm] if limit == 0 else ids[mm][:limit]
                assert np.array_equal(r.column(0), exp)
        with eng.execute(Query("test_1b", conj(Select("age", GT(18)), Select("age", LT(30))), Project(["id", "age"]))) as r:       # C2 on the PFOR table
            assert r.nrows == int(m.sum()) and np.array_equal(r.column(0), ids[m]) and np.array_equal(r.column(1), age[m])
