"""Every kernel route the planner and its switches can choose, against the oracle.

The planner picks the kernels of a query from the table's shape (fill_scan_plan: lane, quad or mini-block filter kernel, pruning,
group emit, scan-emit, prefix pass ...) and the IMM3_* switches of DESIGN §4.7 force the other routes.  Results are bit-identical
on every route (DESIGN §4.2).  Each route below runs a fixed query corpus on small tables written with the product writer and
compares rows, values and order with the oracle; Result.route (imm3_result_route) must show on the route's first query that the
route was actually taken, so a switch that stops working fails here instead of silently testing the default again."""
import re
from collections import namedtuple

import numpy as np
import pytest

import oracle_lib as O
from helpers import conj, oracle_preds
from immutable3_b200 import (EQ, GT, LT, OPEN_NO_STATS, OPEN_NO_TMA, Count, Engine, Max, NoSelect, Project, ProjectAgg, Query,
                             SegmentManager, Select)
from immutable3_b200 import _lib as L
from immutable3_b200.loader import SegmentWriter, synth_write

pytestmark = pytest.mark.gpu


def _wrap(v):
    return ((np.asarray(v, dtype=np.int64) + 2**31) % 2**32 - 2**31).astype(np.int32)


# name -> (id column builder, block rows, blocks per segment, id codec, filter kernel the planner picks for a range on `id`).
# Families pinned from today's thresholds (a 32-block tile of the column in a ring slot: <= ~14 KB lane, <= 40 KB quad, else
# mini-block); at most 10 segments, so canonical order (file-name order) is write order.
TABLES = {
    # dense sorted ids, widths (B, 1, 1, ...): starts just below 2^17 / 2^29 / 2^31 - n put two first-mini-block widths into one
    # tile; every segment ends in a 1-row block
    "d17": (lambda rng: _wrap(np.arange(70_001) + (1 << 17) - 3000), 1024, 14, "PFOR_INT", "lane"),
    "d29": (lambda rng: _wrap(np.arange(70_001) + (1 << 29) - 40_000), 1000, 15, "PFOR_INT", "lane"),
    "d31": (lambda rng: _wrap(np.arange(70_001) + 2**31 - 70_001), 1024, 16, "PFOR_INT", "lane"),
    "s32": (lambda rng: _wrap(np.cumsum(rng.integers(0, 16, 40_000))), 32, 300, "PFOR_INT", "lane"),
    # sorted, deltas of ~4 and ~8 bits: the quad kernel by default
    "b4": (lambda rng: _wrap(np.cumsum(rng.integers(0, 16, 100_000)) - 5_000_000), 1024, 20, "PFOR_INT", "quad"),
    "b8": (lambda rng: _wrap(np.cumsum(rng.integers(0, 256, 100_000)) - 2**30), 1024, 20, "PFOR_INT", "quad"),
    # 12-bit deltas and an unsorted column (every mini-block raw): the mini-block kernel by default
    "b12": (lambda rng: _wrap(np.cumsum(rng.integers(0, 4096, 100_000)) - 2**31 + 5), 1024, 20, "PFOR_INT", "mini"),
    "rnd": (lambda rng: rng.integers(-2**31, 2**31, 50_000).astype(np.int32), 1024, 10, "PFOR_INT", "mini"),
    # narrow deltas with wide jumps, wrapping past 2^31 mid-table, a run of raw mini-blocks; blocks of 1000 rows (var-byte tails)
    "raw": (None, 1000, 12, "PFOR_INT", "quad"),
    # dense-id twin of b4: the row-space pipeline
    "twin": (None, 1024, 20, "DENSE_INT", "dense"),
}
LANE_T, QUAD_T, MINI_T = ["d17", "d29", "d31", "s32"], ["b4", "b8", "raw"], ["b12", "rnd"]
BLOCK_T = LANE_T + QUAD_T + MINI_T
ALL_T = BLOCK_T + ["two", "twin"]


def _raw_ids(rng):
    n = 60_000
    d = rng.choice([0, 1, 2, 3, 1 << 20], size=n, p=[0.1, 0.4, 0.3, 0.19, 0.01]).astype(np.int64)
    v = np.cumsum(d)
    v = v + (2**31 - int(v[n // 2]))
    v[20_000:20_150] = rng.integers(-2**31, 2**31, 150)
    return _wrap(v)


Tab = namedtuple("Tab", "block family queries")


def _corpus(v, block, seg_blocks, ts=None):
    """Named queries of one table: C4 windows whose edges fall on, just before and just after a block boundary and a mini-block
    boundary, one row, an empty window, the whole table, EQ on the extremes, GT / LT alone, a range combined with age < 50,
    age < 50 alone (row-space filter on a block table), no predicate."""
    n, v64 = len(v), v.astype(np.int64)
    seg_rows = block * seg_blocks + 1
    p = seg_rows + 3 * block if n > seg_rows + 6 * block else 3 * block  # a block boundary inside the second segment
    q = p + min(160, block // 2)                                             # a mini-block boundary (block 32: mid-block)
    w = min(2000, n // 8)
    rng_ = lambda lo, hi: conj(Select("id", GT(min(lo, hi))), Select("id", LT(max(lo, hi))))
    qs = {"c4": rng_(int(v64[n // 3]), int(v64[n // 2]))}
    for name, e in (("blk", p), ("mini", q)):
        for d in (-1, 0, 1):
            qs[f"{name}{d:+d}/end"] = rng_(int(v64[e + d - w]), int(v64[e + d]))
            qs[f"{name}{d:+d}/start"] = rng_(int(v64[e + d]) - 1, int(v64[e + d + w]))
    x = int(v64[p])
    qs["one"] = rng_(x - 1, x + 1)
    sv = np.sort(v64)
    gaps = np.flatnonzero(np.diff(sv) >= 2)  # a range between two neighbouring values: not empty by its bounds, no row inside
    lo_, hi_ = int(sv[0]), int(sv[-1])
    qs["empty"] = rng_(int(sv[gaps[0]]), int(sv[gaps[0] + 1])) if len(gaps) else rng_(lo_ - 10, lo_)
    qs["whole"] = conj(Select("id", GT(lo_ - 1)), Select("id", LT(hi_ + 1)))
    qs["eq_min"], qs["eq_max"] = Select("id", EQ(lo_)), Select("id", EQ(hi_))
    qs["gt"], qs["lt"] = Select("id", GT(int(v64[n // 2]))), Select("id", LT(int(v64[n // 2])))
    qs["mixed"] = conj(Select("id", GT(int(v64[n // 4]))), Select("id", LT(int(v64[3 * n // 4]))), Select("age", LT(50)))
    qs["age"] = Select("age", LT(50))
    qs["none"] = NoSelect
    if ts is not None:  # predicates on two encoded columns
        qs["c4_two"] = conj(Select("id", GT(int(v64[n // 4]))), Select("id", LT(int(v64[3 * n // 4]))), Select("ts", GT(int(ts[n // 3]))))
    return qs


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("routes")
    rng = np.random.default_rng(2024)
    tabs = {}
    for name, (make, block, seg, codec, family) in TABLES.items():
        if name == "twin":
            ids = tabs["b4"][1]
        elif name == "raw":
            ids = _raw_ids(rng)
        else:
            ids = make(rng)
        ages = rng.integers(0, 100, size=len(ids)).astype(np.int8)
        if name == "twin":
            ages = tabs["b4"][2]
        with SegmentWriter(d, name, [f"id:{codec}", "age:DENSE_TINYINT"], block, seg) as w:
            w.append(ids, ages)
        tabs[name] = (Tab(block, family, _corpus(ids, block, seg)), ids, ages)
    # two encoded columns (a dense sorted id and a sorted ~6-bit ts) and a dense age
    n = 60_000
    ids = _wrap(np.arange(n) + 1_000_000)
    ts = _wrap(np.cumsum(rng.integers(0, 64, n)) - 7)
    ages = rng.integers(0, 100, size=n).astype(np.int8)
    with SegmentWriter(d, "two", ["id:PFOR_INT", "ts:PFOR_INT", "age:DENSE_TINYINT"], 1024, 18) as w:
        w.append(ids, ts, ages)
    tabs["two"] = (Tab(1024, "lane", _corpus(ids, 1024, 18, ts=ts)), ids, ages)
    memo = {}
    with O.Oracle(d) as orc:
        def expect(table, sel, proj, limit):
            key = (table, sel, tuple(proj), limit)
            if key not in memo:
                memo[key] = orc.query(table, oracle_preds(sel), proj, limit=limit)
            return memo[key]

        yield d, {k: v[0] for k, v in tabs.items()}, expect


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


LANE = r"blocks_filter_lane/w=\d+/s=2"
QUAD = r"blocks_filter_quad/s=\d+"
MINI = r"blocks_filter/s=\d+"
# the default route of a C4 query projecting the encoded column, by the filter kernel the table's shape picks
DEFAULT_C4 = {"lane": rf"^blocks_prune;{LANE};blocks_group_emit/ctas=\d+$", "quad": rf"^blocks_prune;{QUAD};blocks_scan_emit$",
              "mini": rf"^blocks_prune;{MINI};blocks_scan_emit$", "dense": r"^filter\(tma\)/s=2;emit_stream/s=2;emit$"}
UNPRUNED_C4 = {"lane": rf"^{LANE};blocks_group_emit/ctas=\d+$", "quad": rf"^{QUAD};blocks_scan_emit$", "mini": rf"^{MINI};blocks_scan_emit$"}
NO_LANE_C4 = dict(DEFAULT_C4, lane=DEFAULT_C4["quad"])
NO_QUAD_C4 = dict(DEFAULT_C4, lane=DEFAULT_C4["mini"], quad=DEFAULT_C4["mini"])
DENSE_AGE = r"^filter\(tma\)/s=4;"  # age < 50 on the dense twin: 8 KB stages, four of them by default

# (name, environment, imm3_open flags, expected route of the first query: a regex or {filter family: regex}, tables,
#  first query: (corpus name, projection, LIMIT))
Route = namedtuple("Route", "name env flags expect tables first")
C4_ID = ("c4", ["id"], 0)
C4_ID_AGE = ("c4", ["id", "age"], 0)
ROUTES = [
    # lane filter kernel
    Route("lane", {}, 0, DEFAULT_C4, LANE_T + ["two"], C4_ID),
    Route("lane_warps4", {"IMM3_LANE_WARPS": "4"}, 0, r"^blocks_prune;blocks_filter_lane/w=4/s=2;offset_scan;blocks_emit\(blocks\)$", ["d17", "s32"], C4_ID_AGE),
    Route("lane_warps7", {"IMM3_LANE_WARPS": "7"}, 0, r"^blocks_prune;blocks_filter_lane/w=7/s=2;offset_scan;blocks_emit\(blocks\)$", ["d31"], C4_ID_AGE),
    Route("lane_warps4_groupemit", {"IMM3_LANE_WARPS": "4"}, 0, r"^blocks_prune;blocks_filter_lane/w=4/s=2;blocks_group_emit/ctas=\d+$", ["d29"], C4_ID),
    Route("lane_warps8", {"IMM3_LANE_WARPS": "8"}, 0, r"^blocks_prune;blocks_filter_lane/w=8/s=2;blocks_emit\(blocks\)$", ["d17", "d29"], C4_ID_AGE),
    Route("lane_warps16", {"IMM3_LANE_WARPS": "16"}, 0, r"^blocks_prune;blocks_filter_lane/w=16/s=2;blocks_group_emit/ctas=\d+$", ["s32"], C4_ID),
    Route("lane_stages3", {"IMM3_LANE_STAGES": "3"}, 0, r"^blocks_prune;blocks_filter_lane/w=\d+/s=3;blocks_group_emit/ctas=\d+$", ["d17", "s32"], C4_ID),
    Route("lane_stages4", {"IMM3_LANE_STAGES": "4"}, 0, r"^blocks_prune;blocks_filter_lane/w=\d+/s=4;blocks_group_emit/ctas=\d+$", ["d31", "s32"], C4_ID),
    Route("lane_debug256", {"IMM3_DEBUG": "256"}, 0, DEFAULT_C4, ["d17", "s32"], C4_ID),
    Route("lane_debug512", {"IMM3_DEBUG": "512"}, 0, DEFAULT_C4, ["d29", "d31"], C4_ID),
    # emit behind the lane kernel
    Route("ge_ctas1", {"IMM3_GE_CTAS": "1"}, 0, rf"^blocks_prune;{LANE};blocks_group_emit/ctas={{sms1}}$", ["d17", "s32"], C4_ID),
    Route("ge_ctas2", {"IMM3_GE_CTAS": "2"}, 0, rf"^blocks_prune;{LANE};blocks_group_emit/ctas={{sms2}}$", ["d31"], C4_ID),
    Route("ge_ctas4", {"IMM3_GE_CTAS": "4"}, 0, rf"^blocks_prune;{LANE};blocks_group_emit/ctas={{sms4}}$", ["d29"], C4_ID),
    Route("no_groupemit", {"IMM3_NO_GROUPEMIT": "1"}, 0, rf"^blocks_prune;{LANE};blocks_scan_emit$", LANE_T, C4_ID),
    Route("no_scanemit", {"IMM3_NO_SCANEMIT": "1"}, 0, rf"^blocks_prune;{LANE};blocks_emit\(blocks\)$", ["d17", "d31"], C4_ID),
    Route("no_scanemit_scan_kernel", {"IMM3_NO_SCANEMIT": "1", "IMM3_SCAN": "kernel"}, 0, rf"^blocks_prune;{LANE};offset_scan;blocks_emit\(blocks\)$",
          ["d29", "s32"], C4_ID),
    Route("lane_two_columns", {}, 0, rf"^blocks_prune;{LANE};blocks_emit\(blocks\)$", LANE_T, C4_ID_AGE),
    # quad filter kernel
    Route("no_lane", {"IMM3_NO_LANE": "1"}, 0, NO_LANE_C4, ALL_T, C4_ID),
    Route("quad", {}, 0, DEFAULT_C4, QUAD_T, C4_ID),
    Route("quad_stages2", {"IMM3_BLOCKS_STAGES": "2"}, 0, r"^blocks_prune;blocks_filter_quad/s=2;blocks_scan_emit$", QUAD_T, C4_ID),
    Route("quad_stages4", {"IMM3_BLOCKS_STAGES": "4"}, 0, r"^blocks_prune;blocks_filter_quad/s=4;blocks_scan_emit$", ["b4", "raw"], C4_ID),
    Route("quad_stages4_no_lane", {"IMM3_BLOCKS_STAGES": "4", "IMM3_NO_LANE": "1"}, 0, r"^blocks_prune;blocks_filter_quad/s=4;blocks_scan_emit$", ["d17"], C4_ID),
    # mini-block filter kernel
    Route("no_quad", {"IMM3_NO_QUAD": "1"}, 0, NO_QUAD_C4, ALL_T, C4_ID),
    Route("mini", {}, 0, DEFAULT_C4, MINI_T, C4_ID),
    Route("two_encoded_predicates", {}, 0, rf"^blocks_prune;{MINI};blocks_scan_emit$", ["two"], ("c4_two", ["id"], 0)),
    Route("mini_stages2", {"IMM3_BLOCKS_STAGES": "2"}, 0, r"^blocks_prune;blocks_filter/s=2;blocks_scan_emit$", ["b12", "rnd"], C4_ID),
    Route("mini_stages5", {"IMM3_BLOCKS_STAGES": "5"}, 0, r"^blocks_prune;blocks_filter/s=5;blocks_scan_emit$", ["b12", "rnd"], C4_ID),
    Route("mini_stages8", {"IMM3_BLOCKS_STAGES": "8"}, 0, r"^blocks_prune;blocks_filter/s=8;blocks_scan_emit$", ["b12"], C4_ID),
    # pruning off
    Route("no_prune", {"IMM3_NO_PRUNE": "1"}, 0, UNPRUNED_C4, ["d17", "b4", "b12"], C4_ID),
    Route("no_stats", {}, OPEN_NO_STATS, UNPRUNED_C4, ["d31", "b8", "rnd"], C4_ID),
    Route("no_stats_no_lane", {"IMM3_NO_LANE": "1"}, OPEN_NO_STATS, rf"^{QUAD};blocks_scan_emit$", ["s32"], C4_ID),
    # dense predicates on a block table
    Route("hybrid", {}, 0, r"^filter\(tma\)/s=4;blocks_emit\(rowspace\)$", ["d17", "b4", "raw", "s32"], ("age", ["id"], 0)),
    Route("no_hybrid", {"IMM3_NO_HYBRID": "1"}, 0, rf"^{MINI};blocks_scan_emit$", ["d17", "b4", "raw", "s32"], ("age", ["id"], 0)),
    # small LIMIT: prefix pass first
    Route("prefix", {"IMM3_PREFIX_ROWS": "8192"}, 0, r"/prefix", ["b4", "b12", "twin"], ("mixed", ["id", "age"], 33)),
    Route("no_prefix", {"IMM3_PREFIX_ROWS": "8192", "IMM3_NO_PREFIX": "1"}, 0, r"^(?!.*/prefix).", ["b4", "b12", "twin"], ("mixed", ["id", "age"], 33)),
    # single pass
    Route("fused", {"IMM3_PATH": "fused"}, 0, r"^scan_blocks$", BLOCK_T + ["two"], C4_ID),
    # completion / timing: same route, same rows
    Route("no_pdl", {"IMM3_NO_PDL": "1"}, 0, DEFAULT_C4, ["d17", "b4", "b12", "twin"], C4_ID),
    Route("no_publish", {"IMM3_NO_PUBLISH": "1"}, 0, DEFAULT_C4, ["d17", "b4", "twin"], C4_ID),
    Route("eager_times", {"IMM3_EAGER_TIMES": "1"}, 0, DEFAULT_C4, ["d31", "b8", "twin"], C4_ID),
    # dense pipeline (the twin)
    Route("dense", {}, 0, DENSE_AGE + r"emit_stream/s=2;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("filter_stages2", {"IMM3_FILTER_STAGES": "2"}, 0, r"^filter\(tma\)/s=2;emit_stream/s=2;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("filter_stages4", {"IMM3_FILTER_STAGES": "4"}, 0, r"^filter\(tma\)/s=4;emit_stream/s=2;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("filter_stages8", {"IMM3_FILTER_STAGES": "8"}, 0, r"^filter\(tma\)/s=8;emit_stream/s=2;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("emit_stages2", {"IMM3_EMIT_STAGES": "2"}, 0, DENSE_AGE + r"emit_stream/s=2;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("emit_stages3", {"IMM3_EMIT_STAGES": "3"}, 0, DENSE_AGE + r"emit_stream/s=3;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("emit_stages4", {"IMM3_EMIT_STAGES": "4"}, 0, DENSE_AGE + r"emit_stream/s=4;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("emit_stream", {"IMM3_EMIT": "stream"}, 0, DENSE_AGE + r"emit_stream/s=2$", ["twin"], ("age", ["id", "age"], 0)),
    Route("emit_gather", {"IMM3_EMIT": "gather"}, 0, DENSE_AGE + r"emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("emit_both", {"IMM3_EMIT": "both"}, 0, DENSE_AGE + r"emit_stream/s=2;emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("no_emit_stream", {"IMM3_NO_EMIT_STREAM": "1"}, 0, DENSE_AGE + r"emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("emit_general", {"IMM3_EMIT_GENERAL": "1"}, 0, DENSE_AGE + r"emit_stream/s=2;emit_general$", ["twin"], ("age", ["id", "age"], 0)),
    Route("no_tma", {}, OPEN_NO_TMA, r"^filter\(direct\);emit$", ["twin"], ("age", ["id", "age"], 0)),
    Route("no_tma_blocks", {}, OPEN_NO_TMA, r"^filter\(direct\);blocks_emit\(rowspace\)$", ["d29", "b8"], ("age", ["id"], 0)),
    Route("keep_l2_0", {"IMM3_KEEP_L2_MB": "0"}, 0, r"^filter\(tma\)/s=2;emit_stream/s=2;emit$", ["twin"], C4_ID),
]
PROJS = (["id"], ["id", "age"])
SEEN = {}  # route name -> the routes its queries took


def _limits(count):
    return sorted({0, 1, 33, count // 2 + 17, count, count + 1})


def _check_launches(got, what):
    """kernel_launches counts the route's entries."""
    r = got.route
    assert got.kernel_launches == (len(r.split(";")) if r else 0), (what, r, got.kernel_launches)


def _run(eng, expect, table, sel, proj, limit, what):
    exp = expect(table, sel, proj, limit)
    with eng.execute(Query(table, sel, Project(proj, limit))) as got:
        _check_launches(got, what)
        assert got.nrows == exp.nrows, (what, table, sel, proj, limit, got.route, got.nrows, exp.nrows)
        for c in range(len(proj)):
            a, b = got.column(c), exp.columns[c]
            if not np.array_equal(a, b):
                bad = int(np.flatnonzero(a != b)[0])
                raise AssertionError(f"{what} {table} {sel} {proj} limit {limit} ({got.route}): column {proj[c]} differs first at row {bad}: "
                                     f"got {a[bad]!r} want {b[bad]!r}")
        return got.route


@pytest.mark.parametrize("route", ROUTES, ids=[r.name for r in ROUTES])
def test_route_matches_the_oracle(world, route, monkeypatch):
    d, tabs, expect = world
    for k, v in route.env.items():
        monkeypatch.setenv(k, v)
    sms = _sms()
    seen = SEEN.setdefault(route.name, set())
    with SegmentManager(d, flags=route.flags) as sm:
        eng = Engine(sm)
        for table in route.tables:
            t = tabs[table]
            want = route.expect[t.family] if isinstance(route.expect, dict) else route.expect
            want = want.replace("{sms1}", str(sms)).replace("{sms2}", str(2 * sms)).replace("{sms4}", str(4 * sms))
            key, proj0, limit0 = route.first
            got = _run(eng, expect, table, t.queries[key], proj0, limit0, route.name)
            print(f"{route.name:26s} {table:5s} {got}")
            assert re.search(want, got), f"{route.name} on {table}: route {got!r} does not match {want!r}"
            seen.add(got)
            for name, sel in t.queries.items():
                for proj in PROJS:
                    count = expect(table, sel, proj, 0).nrows
                    for limit in _limits(count):
                        seen.add(_run(eng, expect, table, sel, proj, limit, f"{route.name}/{name}"))


KERNELS = {"blocks_filter_lane", "blocks_filter_quad", "blocks_filter", "blocks_prune", "blocks_group_emit", "blocks_scan_emit",
           "blocks_emit(rowspace)", "blocks_emit(blocks)", "scan_blocks", "offset_scan", "emit_stream", "emit", "emit_general",
           "select_all", "filter(tma)", "filter(direct)"}


def test_the_matrix_reaches_every_kernel():
    """Across the whole matrix every kernel of the single-GPU scan path ran at least once (the count exchange is
    test_gpu_dist.py's)."""
    if len(SEEN) < len(ROUTES):
        pytest.skip("needs every route of this module to have run first")
    names = {k.split("/")[0] for routes in SEEN.values() for r in routes for k in r.split(";") if k}
    print("kernels seen:", " ".join(sorted(names)))
    assert KERNELS <= names, sorted(KERNELS - names)


def test_aggregate_routes(world):
    """imm3_query_agg reports its launches too: the dense aggregation kernel, and the block-decoding one for an encoded MIN / MAX
    input, each with the <NG, NA> instantiation it ran."""
    d, tabs, expect = world
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        with eng.execute(Query("twin", Select("age", LT(50)), ProjectAgg([Count("id")]))) as r:
            assert re.search(r"^agg_init;filter\(tma\)/s=4;agg<0,1>;agg_compact$", r.route), r.route
            assert r.kernel_launches == 4 and int(r.column(0)[0]) == expect("twin", Select("age", LT(50)), ["id"], 0).nrows
        with eng.execute(Query("b4", NoSelect, ProjectAgg([Max("id"), Count("age")], ["age"]))) as r:
            assert re.search(r"^agg_init;select_all;agg_blocks<1,2>;agg_compact$", r.route), r.route
            _check_launches(r, "agg_blocks")


def test_block_routes_at_40m_rows(tmp_path_factory, monkeypatch):
    """The block routes at a size the oracle cannot handle: a 40 M-row synthetic table whose id is in the sorted-int codec
    (the 1 B-row table's shape), written once; the switches are read per query, OPEN_NO_STATS needs a second open.  Checked
    against numpy on the files."""
    d = tmp_path_factory.mktemp("routes40m")
    n = 40_000_000
    synth_write(d, "big", n, id_codec=L.CODEC_PFOR_INT)
    nseg = (n + 1024 * 1000) // (1024 * 1000 + 1)
    order = sorted(range(nseg), key=lambda i: f"id_{i}.dat")
    per = 1024 * 1000 + 1
    ids = np.concatenate([np.arange(i * per, min(n, (i + 1) * per), dtype=np.int32) for i in order])
    age = np.concatenate([np.fromfile(d / "big" / f"age_{i}.dat", np.int8) for i in order])
    lo, hi = n // 2 - n // 200, n // 2 + n // 200
    b = 4 * per  # a segment boundary (segment 4 follows segment 39 in file-name order)
    cases = [(conj(Select("id", GT(lo)), Select("id", LT(hi))), ["id"], 0),
             (conj(Select("id", GT(lo)), Select("id", LT(hi))), ["id"], 123_457),
             (conj(Select("id", GT(b - 700)), Select("id", LT(b + 1500))), ["id", "age"], 0),
             (conj(Select("id", GT(n - 3000)), Select("id", LT(n + 5))), ["id"], 1000),
             (Select("id", EQ(b - 1)), ["id", "age"], 0)]
    # (environment, open flags, filter part of the route, emit kernel when `id` alone is projected); with `id, age` projected
    # the general block emit kernel runs behind any of them
    lane = r"blocks_filter_lane/w=\d+/s=2;"
    routes = [({}, 0, r"^blocks_prune;" + lane, r"blocks_group_emit/ctas=\d+$"),
              ({"IMM3_NO_LANE": "1"}, 0, r"^blocks_prune;blocks_filter_quad/s=\d+;", r"blocks_scan_emit$"),
              ({"IMM3_NO_QUAD": "1"}, 0, r"^blocks_prune;blocks_filter/s=\d+;", r"blocks_scan_emit$"),
              ({"IMM3_NO_GROUPEMIT": "1"}, 0, r"^blocks_prune;" + lane, r"blocks_scan_emit$"),
              ({"IMM3_NO_PRUNE": "1"}, 0, "^" + lane, r"blocks_group_emit/ctas=\d+$"),
              ({}, OPEN_NO_STATS, "^" + lane, r"blocks_group_emit/ctas=\d+$")]
    sm = None
    try:
        for env, flags, filt, emit1 in routes:
            if sm is None or sm.flags != flags:
                if sm is not None:
                    sm.close()
                sm = SegmentManager(d, flags=flags)
            for k in ("IMM3_NO_LANE", "IMM3_NO_QUAD", "IMM3_NO_GROUPEMIT", "IMM3_NO_PRUNE"):
                monkeypatch.delenv(k, raising=False)
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            eng = Engine(sm)
            for sel, proj, limit in cases:
                lo_, hi_ = sel.op1.cond.gt if hasattr(sel, "op1") else None, sel.op2.cond.lt if hasattr(sel, "op2") else None
                m = (ids > lo_) & (ids < hi_) if lo_ is not None else ids == sel.cond.eq
                with eng.execute(Query("big", sel, Project(proj, limit))) as r:
                    if limit == 0:
                        # no LIMIT: one launch sequence, exactly the route of the switch
                        want = filt + (emit1 if len(proj) == 1 else r"blocks_emit\(blocks\)$")
                        assert re.search(want, r.route), (env, flags, sel, r.route, want)
                    want_ids = ids[m][:limit] if limit else ids[m]
                    assert r.nrows == len(want_ids), (env, flags, sel, limit, r.route, r.nrows, len(want_ids))
                    assert np.array_equal(r.column(0), want_ids), (env, flags, sel, limit, r.route)
                    if len(proj) > 1:
                        assert np.array_equal(r.column(1), age[m][:limit] if limit else age[m]), (env, flags, sel, limit, r.route)
    finally:
        if sm is not None:
            sm.close()
