"""Real OR on the row-space pipeline (imm3_query_begin_dnf without IMM3_DNF_ENCODED_FILTER) across the planner's routes and
switches, the two-phase LIMIT, ranks and a 40 M-row table, against select_tree_ref.eval_tree.

Every term of such a disjunction runs filter_kernel over the same selection bitmap: the second and later terms OR their rows
into it (ScanPlan::or_accumulate), each pass rewrites the span and tile counts of the union so far, and only the last pass
may turn the tile counts into offsets (launch_row_space_filter).  The expected rows here come from walking the select tree itself
with numpy, not from select_dnf's expansion, so a wrong expansion cannot move the expected and the actual rows together.

As in test_gpu_routes.py, a route's first query must show in Result.route that the route's switch applied, and every query
must report one launch per route entry.  In each LIMIT phase every conjunction that survives narrowing launches exactly one
filter kernel."""
import os
import re
import sys
from collections import namedtuple

import numpy as np
import pytest

import oracle_lib as O
from helpers import STATES, make_table
from immutable3_b200 import (EQ, GT, LT, OPEN_FORCE_BLOCKS, OPEN_HOST_ONLY, OPEN_NO_TMA, And, Engine, Imm3Error, Match, NoSelect, Or,
                             Project, Query, SegmentManager, Select, select_dnf)
from immutable3_b200 import _lib as L
from select_tree_ref import can_hold, canonical_columns, eval_tree, expected_rows, random_tree

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

NAMES = np.array([b"alice", b"bobby", b"carol", b"dave_", b"erin#"], "S5")
CODES = np.array([b"k001", b"k002", b"zz99", b"abcd"], "S4")
COLS = ["id", "state", "age", "score", "name", "code", "pos"]

# name -> (rows, block rows, blocks per segment, id codec, id order, family).  Every table also has score (DENSE_INT), name
# (DENSE_STRING(5)), code (DENSE_STRING(4)) and pos (DENSE_INT, the write-order row number): a term on score, name and code
# stages 13 bytes per row, more than a 56 KB TMA stage of 8192 rows holds, so it loads directly beside a staged term on age.
# Even make_table seeds: ages 0 .. 99.
TABLES = {
    "r": (50_003, 1024, 7, "DENSE_INT", "sorted", "dense"),      # 7 segments; 7 tiles of 8192 rows, the last ragged
    "x2": (16_384, 1024, 20, "DENSE_INT", "sorted", "dense"),     # exactly two tiles, one segment
    "one": (1, 1024, 20, "DENSE_INT", "sorted", "dense"),
    "many": (30_000, 100, 10, "DENSE_INT", "random", "dense"),   # 30 segments: canonical (file-name) order is not write order
    "p1024": (40_000, 1024, 3, "PFOR_INT", "steps", "pfor"),     # sorted-int-codec id: dense predicates take the hybrid
    "p1000": (30_001, 1000, 3, "PFOR_INT", "sorted", "pfor"),
    "p32": (5_001, 32, 40, "PFOR_INT", "sorted", "pfor"),
}
DENSE_T, PFOR_T = ["r", "x2", "one", "many"], ["p1024", "p1000", "p32"]


def extra_cols(n, rng):
    return [("score:DENSE_INT", rng.integers(-1000, 1000, n).astype(np.int32)),
            ("name:DENSE_STRING:size=5", NAMES[rng.integers(0, 5, n)]),
            ("code:DENSE_STRING:size=4", CODES[rng.integers(0, 4, n)]),
            ("pos:DENSE_INT", np.arange(n, dtype=np.int32))]


def age(op, v):
    return Select("age", op(v))


def corpus(cols, dense_id):
    """Named disjunctions over the dense columns of a table (canonical columns `cols`)."""
    n = len(cols["pos"])
    at = lambda i: int(cols["pos"][min(max(i, 0), n - 1)])                 # pos of canonical row i
    pos = lambda i: Select("pos", EQ(at(i)))
    x = And(age(GT, 30), age(LT, 70))
    qs = {
        "two": Or(age(LT, 10), age(GT, 90)),
        "three": Or(And(age(GT, 20), age(LT, 30)), Or(Select("score", GT(900)), age(EQ, 55))),
        "match": Or(Select("state", Match(["CA", "NY"])), Select("name", Match(["alice", "erin#"]))),
        # 100 literals of 5 bytes: 500 of the 512 bytes of the literal pool
        "pool": Or(Select("name", Match(["bobby"] + [f"x{i:04d}" for i in range(99)])), And(Select("state", Match(STATES[:40])), age(LT, 7))),
        "staged_direct": Or(age(LT, 5), And(Select("score", GT(0)), And(Select("name", Match(["carol", "dave_"])), Select("code", Match(["k001", "abcd"]))))),
        "direct_staged": Or(And(Select("score", LT(-500)), And(Select("name", Match(["alice"])), Select("code", Match(["zz99"])))), age(GT, 95)),
        "overlap": Or(And(age(GT, 10), age(LT, 60)), And(age(GT, 40), age(LT, 80))),
        "nested": Or(And(age(GT, 10), age(LT, 80)), And(age(GT, 30), age(LT, 40))),
        "same": Or(x, x),
        "never_first": Or(Select("score", GT(5000)), age(LT, 20)),        # the first term runs and holds nowhere
        "narrowed_first": Or(age(GT, -129), age(LT, 20)),                 # -129 narrows to 127: dropped before any kernel
        "true_first": Or(age(GT, -1), Select("state", Match(["CA"]))),    # a term that holds on every row
        "true_last": Or(Select("state", Match(["CA"])), age(GT, -1)),
        "noselect": Or(age(LT, 3), NoSelect),                             # a conjunction without predicates: every row
        "sixteen": And(Or(age(LT, 20), Select("state", Match(["CA", "TX"]))),
                       And(Or(Select("score", GT(500)), Select("name", Match(["carol"]))),
                           And(Or(age(GT, 50), Select("code", Match(["k001"]))), Or(Select("score", LT(-700)), age(EQ, 33))))),
        "none": Or(Select("state", Match(["ZZ"])), Select("score", GT(5000))),
        "early": Or(pos(0), And(age(LT, 50), Select("state", Match(["CA"])))),
        "late": Or(pos(n - 1), Or(pos(n - 5), pos(3 * n // 4))),          # rows only far behind the first 8192
        "split": Or(pos(3), Or(pos(n - 1), pos(n - 2))),                  # one row in front, two far behind
        # the second row lies in the first 8192-row tile but behind the 8 blocks of a block table's prefix phase
        "edge": Or(pos(0), pos(min(8000, n - 1))),
    }
    if dense_id:
        ids = np.sort(cols["id"].astype(np.int64))
        q = lambda f: int(ids[int(f * (n - 1))])
        qs["id"] = Or(Select("id", LT(q(0.1))), And(Select("id", GT(q(0.6))), age(LT, 50)))
    return qs


class Tab:
    def __init__(self, name, family, cols, nblocks):
        self.name, self.family, self.cols, self.nblocks = name, family, cols, nblocks
        self.queries = corpus(cols, family == "dense")
        self._masks = {}

    def mask(self, key):
        if key not in self._masks:
            self._masks[key] = eval_tree(self.cols, self.queries[key])
        return self._masks[key]


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("real_or_routes")
    rng = np.random.default_rng(31)
    for i, (name, (n, block, seg, codec, mode, fam)) in enumerate(TABLES.items()):
        make_table(d, name, n, block, seg, seed=2 * i + 2, id_codec=codec, id_mode=mode, extra_cols=extra_cols(n, rng))
    with O.Oracle(d) as orc, SegmentManager(d, flags=OPEN_HOST_ONLY) as info:
        tabs = {name: Tab(name, TABLES[name][5], canonical_columns(orc, name, COLS), info.getTable(name).nblocks) for name in TABLES}
    yield d, tabs


def live_terms(sel, cols):
    """Filter kernels one LIMIT phase of the disjunction launches: one per conjunction that survives narrowing (a conjunction
    without predicates makes the whole query one select_all)."""
    terms = select_dnf(sel)
    if any(len(t) == 0 for t in terms):
        return 1
    return sum(1 for t in terms if can_hold(t, cols))


def phases(route):
    """(filter launches of the prefix phase, ... of the whole-table phase)."""
    parts = route.split(";") if route else []
    filt = lambda p: p.startswith(("filter(", "select_all", "blocks_filter", "scan_blocks"))
    a = sum(1 for p in parts if p.endswith("/prefix") and filt(p))
    b = sum(1 for p in parts if not p.endswith("/prefix") and filt(p))
    return a, b


def run(eng, table, cols, sel, proj, limit, what, mask=None, encoded=False):
    """The disjunction against eval_tree (rows, values, order); checks the launch count and the filter launches per phase;
    returns the route."""
    mask = eval_tree(cols, sel) if mask is None else mask
    want = expected_rows(cols, mask, proj, limit)
    count = int(mask.sum()) if limit <= 0 else min(int(mask.sum()), limit)
    with eng.execute(Query(table, sel, Project(proj, limit)), real_or=True, encoded_filter=encoded) as got:
        r = got.route
        assert got.kernel_launches == (len(r.split(";")) if r else 0), (what, table, r, got.kernel_launches)
        assert got.nrows == count, (what, table, sel, proj, limit, r, got.nrows, count)
        for c in range(len(proj)):
            a, b = got.column(c), want[c]
            if not np.array_equal(a, b):
                bad = int(np.flatnonzero(a != b)[0])
                raise AssertionError(f"{what} {table} {sel} {proj} limit {limit} ({r}): column {proj[c]} differs first at row {bad}: "
                                     f"got {a[bad]!r} want {b[bad]!r}")
    live = live_terms(sel, cols)
    fa, fb = phases(r)
    if live == 0:
        assert r == "", (what, table, sel, r)
    else:
        assert fa in (0, live) and fb in (0, live) and fa + fb > 0, (what, table, sel, limit, r, live)
        assert ("/prefix" in r) == (fa > 0), (what, table, sel, limit, r)
    return r


F4 = r"filter\(tma\)/s=4;filter\(tma\)/s=4;"
DEFAULT = {"dense": rf"^{F4}emit_stream/s=2;emit$", "pfor": rf"^{F4}blocks_emit\(rowspace\)$"}


def stages(s):
    f = rf"filter\(tma\)/s={s};filter\(tma\)/s={s};"
    return {"dense": rf"^{f}emit_stream/s=2;emit$", "pfor": rf"^{f}blocks_emit\(rowspace\)$"}


# (name, environment, imm3_open flags, expected route of the first query: a regex or {family: regex}, tables,
#  first query: (corpus name, projection, LIMIT))
Route = namedtuple("Route", "name env flags expect tables first")
FIRST = ("two", ["id", "age"], 0)
LATE1 = ("late", ["id", "age"], 1)
ROUTES = [
    Route("default", {}, 0, DEFAULT, DENSE_T + PFOR_T, FIRST),
    Route("filter_stages2", {"IMM3_FILTER_STAGES": "2"}, 0, stages(2), ["r", "many", "p1024"], FIRST),
    Route("filter_stages4", {"IMM3_FILTER_STAGES": "4"}, 0, stages(4), ["x2", "p32"], FIRST),
    Route("filter_stages8", {"IMM3_FILTER_STAGES": "8"}, 0, stages(8), ["r", "one", "p1000"], FIRST),
    Route("no_tma", {}, OPEN_NO_TMA, {"dense": r"^filter\(direct\);filter\(direct\);emit$",
                                     "pfor": r"^filter\(direct\);filter\(direct\);blocks_emit\(rowspace\)$"}, ["r", "x2", "many", "p1000"], FIRST),
    Route("scan_kernel", {"IMM3_SCAN": "kernel"}, 0, {"dense": rf"^{F4}offset_scan;emit_stream/s=2;emit$",
                                                     "pfor": rf"^{F4}offset_scan;blocks_emit\(rowspace\)$"}, ["r", "one", "many", "p32"], FIRST),
    Route("scan_inline", {"IMM3_SCAN": "inline"}, 0, DEFAULT, ["r", "p1024"], FIRST),
    Route("emit_stream", {"IMM3_EMIT": "stream"}, 0, rf"^{F4}emit_stream/s=2$", ["r", "many"], FIRST),
    Route("emit_gather", {"IMM3_EMIT": "gather"}, 0, rf"^{F4}emit$", ["r", "x2"], FIRST),
    Route("emit_both", {"IMM3_EMIT": "both"}, 0, rf"^{F4}emit_stream/s=2;emit$", ["r", "many"], FIRST),
    Route("no_emit_stream", {"IMM3_NO_EMIT_STREAM": "1"}, 0, rf"^{F4}emit$", ["r", "one"], FIRST),
    Route("emit_stages3", {"IMM3_EMIT_STAGES": "3"}, 0, rf"^{F4}emit_stream/s=3;emit$", ["r"], FIRST),
    Route("emit_stages4", {"IMM3_EMIT_STAGES": "4"}, 0, rf"^{F4}emit_stream/s=4;emit$", ["x2"], FIRST),
    Route("emit_general", {"IMM3_EMIT_GENERAL": "1"}, 0, rf"^{F4}emit_stream/s=2;emit_general$", ["r", "many"], FIRST),
    Route("no_pdl", {"IMM3_NO_PDL": "1"}, 0, DEFAULT, ["r", "many", "p1024"], FIRST),
    Route("no_publish", {"IMM3_NO_PUBLISH": "1"}, 0, DEFAULT, ["r", "p1000"], FIRST),
    Route("eager_times", {"IMM3_EAGER_TIMES": "1"}, 0, DEFAULT, ["x2", "p32"], FIRST),
    Route("keep_l2_0", {"IMM3_KEEP_L2_MB": "0"}, 0, DEFAULT, ["r", "p1024"], FIRST),
    # the row-space filter and the block emit kernel on dense tables
    Route("force_blocks", {}, OPEN_FORCE_BLOCKS, rf"^{F4}blocks_emit\(rowspace\)$", ["r", "x2", "many"], FIRST),
    # small LIMIT: the prefix phase first (8192 rows on a dense table, 8 blocks on a block table)
    Route("prefix", {"IMM3_PREFIX_ROWS": "8192"}, 0, r"/prefix", ["r", "x2", "many", "p1024", "p1000", "p32"], LATE1),
    Route("no_prefix", {"IMM3_PREFIX_ROWS": "8192", "IMM3_NO_PREFIX": "1"}, 0, r"^(?!.*/prefix).", ["r", "many", "p1024"], LATE1),
]
PROJS = (["id", "age"], ["name", "id", "state", "age", "score", "id"])  # (six columns, one 5 bytes wide: the general emit)
SEEN = {}      # route name -> the routes its queries took
MULTI = set()  # routes of queries whose tree expands to two or more conjunctions


def _limits(count):
    return sorted({0, 1, 33, count // 2 + 17, count, count + 1} | {k for k in (8191, 8192, 8193) if k <= count})


def prefix_applies(t, limit):
    """Whether a LIMIT takes the prefix phase with IMM3_PREFIX_ROWS=8192 (fill_scan_plan)."""
    if not 1 <= limit <= (1 << 20):
        return False
    rows = max(8192, 64 * limit)
    if t.family == "dense":
        return (rows + 8191) // 8192 * 8192 * 2 <= len(t.cols["pos"])
    return (rows + 1023) // 1024 * 2 <= t.nblocks


@pytest.mark.parametrize("route", ROUTES, ids=[r.name for r in ROUTES])
def test_route_matches_the_tree(world, route, monkeypatch):
    d, tabs = world
    for k, v in route.env.items():
        monkeypatch.setenv(k, v)
    seen = SEEN.setdefault(route.name, set())
    prefix_on = "IMM3_PREFIX_ROWS" in route.env and "IMM3_NO_PREFIX" not in route.env
    with SegmentManager(d, flags=route.flags) as sm:
        eng = Engine(sm)
        for name in route.tables:
            t = tabs[name]
            want = route.expect[t.family] if isinstance(route.expect, dict) else route.expect
            key, proj0, limit0 = route.first
            got = run(eng, name, t.cols, t.queries[key], proj0, limit0, route.name, t.mask(key))
            print(f"{route.name:16s} {name:6s} {got}")
            assert re.search(want, got), f"{route.name} on {name}: route {got!r} does not match {want!r}"
            seen.add(got)
            for key, sel in t.queries.items():
                m = t.mask(key)
                multi = len(select_dnf(sel)) >= 2
                for proj in PROJS:
                    for limit in _limits(int(m.sum())):
                        r = run(eng, name, t.cols, sel, proj, limit, f"{route.name}/{key}", m)
                        seen.add(r)
                        if multi:
                            MULTI.add(r)
                        if "IMM3_NO_PREFIX" in route.env:
                            assert "/prefix" not in r, (route.name, name, key, limit, r)
                        if prefix_on and prefix_applies(t, limit) and live_terms(sel, t.cols) > 0:
                            fa, fb = phases(r)
                            assert fa > 0, (route.name, name, key, limit, r)
                            if int(m[:256].sum()) >= limit:     # phase A (at least 256 rows) fills the LIMIT
                                assert fb == 0, (route.name, name, key, limit, r)
                            if key == "late" and m.any():     # no row in phase A: phase B runs
                                assert fb > 0, (route.name, name, key, limit, r)


KERNELS = {"filter(tma)", "filter(direct)", "select_all", "offset_scan", "emit_stream", "emit", "emit_general", "blocks_emit(rowspace)"}


def test_the_matrix_reaches_every_kernel():
    """Across the matrix every kernel of the row-space disjunction ran in a query of two or more conjunctions.  (select_all
    only where a conjunction has no predicate: narrowing never removes a predicate, so a term that holds everywhere still
    runs the filter kernel.)"""
    if len(SEEN) < len(ROUTES):
        pytest.skip("needs every route of this module to have run first")
    names = {k.split("/")[0] for r in MULTI for k in r.split(";") if k}
    print("kernels seen:", " ".join(sorted(names)))
    assert KERNELS <= names, sorted(KERNELS - names)


def test_emit_hint_learned_on_another_shape(world):
    """The stream-or-gather emit hint is keyed by the first term's filters and the projection, so a disjunction shares it with
    its first term alone.  Whichever single emit kernel the hint picks, the disjunction's rows must be right."""
    d, tabs = world
    t = tabs["r"]
    proj_a, proj_b = ["id", "age"], ["age", "state"]
    sparse_dnf = Or(age(LT, 3), Select("state", Match(["CA"])))
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        # a sparse conjunction teaches "gather only"; the dense disjunction that starts with a term of its shape gathers
        assert run(eng, "r", t.cols, age(EQ, 7), proj_a, 0, "hint").endswith("emit_stream/s=2;emit")   # (no hint yet: both)
        assert re.search(r"^filter\(tma\)/s=4;emit$", run(eng, "r", t.cols, age(EQ, 7), proj_a, 0, "hint"))
        r = run(eng, "r", t.cols, Or(age(EQ, 7), age(GT, 5)), proj_a, 0, "hint")
        assert re.search(rf"^{F4}emit$", r), r
        # the reverse: a dense conjunction teaches "stream only"; a sparse disjunction of that shape streams
        run(eng, "r", t.cols, age(GT, 5), proj_b, 0, "hint")
        assert re.search(r"^filter\(tma\)/s=4;emit_stream/s=\d$", run(eng, "r", t.cols, age(GT, 5), proj_b, 0, "hint"))
        r = run(eng, "r", t.cols, sparse_dnf, proj_b, 0, "hint")
        assert re.search(r"^filter\(tma\)/s=4;filter\(tma\)/s=\d;emit_stream/s=\d$", r), r
        for limit in (1, 33, 1000):
            run(eng, "r", t.cols, sparse_dnf, proj_b, limit, "hint")
            run(eng, "r", t.cols, Or(age(EQ, 7), age(GT, 5)), proj_a, limit, "hint")


def test_refusals_leave_the_handle_working(world, monkeypatch):
    """The single-pass kernel (IMM3_PATH=fused under OPEN_FORCE_BLOCKS) and the block filter kernels (IMM3_NO_HYBRID on a
    block table) cannot accumulate a disjunction: refused with IMM3_ERR_UNSUPPORTED, and the next query on the handle runs."""
    d, tabs = world
    two = tabs["r"].queries["two"]
    with SegmentManager(d, flags=OPEN_FORCE_BLOCKS) as sm:
        eng = Engine(sm)
        monkeypatch.setenv("IMM3_PATH", "fused")
        with pytest.raises(Imm3Error) as e:
            eng.execute(Query("r", two, Project(["id", "age"])), real_or=True)
        assert e.value.status == L.ERR_UNSUPPORTED
        monkeypatch.delenv("IMM3_PATH")
        assert run(eng, "r", tabs["r"].cols, two, ["id", "age"], 0, "after fused").endswith("blocks_emit(rowspace)")
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        monkeypatch.setenv("IMM3_NO_HYBRID", "1")
        for name in PFOR_T:
            with pytest.raises(Imm3Error) as e:
                eng.execute(Query(name, two, Project(["id", "age"])), real_or=True)
            assert e.value.status == L.ERR_UNSUPPORTED
        monkeypatch.delenv("IMM3_NO_HYBRID")
        for name in PFOR_T:
            assert run(eng, name, tabs[name].cols, two, ["id", "age"], 33, "after no_hybrid").endswith("blocks_emit(rowspace)")


def test_blocks_of_4096_rows(tmp_path_factory):
    """A block table whose blocks hold more than 1024 rows: a disjunction of dense predicates that projects only dense
    columns runs the dense pipeline; projecting the encoded column needs the single-pass kernel, which cannot accumulate a
    disjunction, so it is refused (IMM3_ERR_UNSUPPORTED)."""
    d = tmp_path_factory.mktemp("or4096")
    rng = np.random.default_rng(9)
    n = 20_000
    make_table(d, "b", n, 4096, 2, seed=2, id_codec="PFOR_INT", id_mode="steps", extra_cols=extra_cols(n, rng))
    with O.Oracle(d) as orc, SegmentManager(d) as sm:
        cols = canonical_columns(orc, "b", COLS)
        eng = Engine(sm)
        qs = corpus(cols, False)
        for key in ("two", "staged_direct", "sixteen", "split"):
            for limit in (0, 1, 33, 5000):
                r = run(eng, "b", cols, qs[key], ["age", "state", "pos"], limit, "4096")
                assert "blocks" not in r, r
            with pytest.raises(Imm3Error) as e:
                eng.execute(Query("b", qs[key], Project(["id", "age"])), real_or=True)
            assert e.value.status == L.ERR_UNSUPPORTED
        run(eng, "b", cols, qs["match"], ["pos"], 0, "4096 after refusal")


# ---- seeded random disjunctions ------------------------------------------------------------------------------------------

TAGS = np.array([b"aaa", b"abc", b"zzz", b"q_q"], "S3")
SWITCHES = [({}, 0), ({"IMM3_FILTER_STAGES": "2"}, 0), ({"IMM3_FILTER_STAGES": "8"}, 0), ({"IMM3_SCAN": "kernel"}, 0), ({"IMM3_EMIT": "gather"}, 0),
            ({"IMM3_EMIT": "stream"}, 0), ({"IMM3_EMIT_GENERAL": "1"}, 0), ({}, OPEN_NO_TMA), ({"IMM3_PREFIX_ROWS": "8192"}, 0),
            ({"IMM3_NO_PDL": "1", "IMM3_NO_PUBLISH": "1"}, 0), ({"IMM3_NO_EMIT_STREAM": "1", "IMM3_EMIT_STAGES": "3"}, 0)]


def refusal(terms, cols, proj, encoded, pfor, block, max_block_rows):
    """The status imm3_query_begin_dnf[_ext] returns for these conjunctions, or None if it runs.  Fewer than two surviving
    conjunctions are a plain conjunction (every route); otherwise every surviving term must run on the row space - unless
    `encoded` and a term tests the encoded id: then every term runs the block filter front, for blocks of at most 1024 rows."""
    if any(len(t) == 0 for t in terms):
        return None
    live = [t for t in terms if can_hold(t, cols)]
    if len(live) <= 1:
        return None
    on_id = lambda t: pfor and any(leaf.col == "id" for leaf in t)
    if encoded and any(on_id(t) for t in live):
        return L.ERR_UNSUPPORTED if max(max_block_rows, block) > 1024 else None
    for t in live:
        if on_id(t) or (pfor and "id" in proj and max_block_rows > 1024):   # block filter kernels / the single-pass kernel
            return L.ERR_UNSUPPORTED
    return None


@pytest.mark.parametrize("seed", range(12))
def test_random_disjunctions(tmp_path_factory, monkeypatch, seed):
    """Random table shape, select tree (<= 16 conjunctions over id, age, state and a 3-byte string column), projection with
    duplicates, LIMIT and one switch set of the matrix; each query with and without encoded_filter, against eval_tree or the
    refusal the planner's rules give."""
    seed += int(os.environ.get("IMM3_TEST_SEED_BASE", "0"))  # (stress runs: other seeds without editing the file)
    rng = np.random.default_rng(4000 + seed)
    d = tmp_path_factory.mktemp(f"ornd{seed}")
    nrows = int(rng.choice([1, 31, 8191, 8192, 8193, 40_000, 150_000]))
    block = int(rng.choice([8, 32, 100, 1000, 1024, 4096]))
    nseg = int(rng.integers(1, 41))
    rows_per_seg = -(-nrows // nseg)
    seg_blocks = max(1, -(-rows_per_seg // block))  # (a segment holds seg_blocks * block + 1 rows)
    pfor = rng.random() < 0.5
    mode = str(rng.choice(["sorted", "steps", "random"]))
    make_table(d, "t", nrows, block, seg_blocks, seed=int(rng.integers(0, 100)), id_codec="PFOR_INT" if pfor else "DENSE_INT", id_mode=mode,
               extra_cols=[("tag:DENSE_STRING:size=3", TAGS[rng.integers(0, 4, nrows)])])
    env, flags = SWITCHES[int(rng.integers(0, len(SWITCHES)))]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    names = ["id", "state", "age", "tag"]
    with O.Oracle(d) as orc:
        cols = canonical_columns(orc, "t", names)
    ids = cols["id"].astype(np.int64)

    def leaf(rng):
        k = int(rng.integers(0, 8))
        if k == 0:
            return age(GT, float(rng.integers(-140, 140)))
        if k == 1:
            return age(LT, float(rng.integers(-140, 140)) + 0.5)
        if k == 2:
            return age(EQ, float(cols["age"][int(rng.integers(0, nrows))]))
        if k in (3, 4):
            q = float(np.quantile(ids, rng.random()))
            return Select("id", GT(q)) if k == 3 else Select("id", LT(q))
        if k == 5:
            return Select("state", Match([str(s) for s in rng.choice(STATES, size=int(rng.integers(1, 8)))]))
        if k == 6:
            return Select("tag", Match([v.decode() for v in rng.choice(TAGS, size=int(rng.integers(1, 3)))] + (["ab"] if rng.random() < 0.3 else [])))
        return Select("age", GT(float(rng.integers(-60, 60)))) if rng.random() < 0.5 else Select("age", LT(float(rng.integers(-60, 60))))

    ran = refused = 0
    with SegmentManager(d, flags=flags) as sm:
        eng = Engine(sm)
        for qi in range(12):
            tree = random_tree(rng, leaf)
            terms = select_dnf(tree)
            proj = [str(c) for c in rng.choice(names, size=int(rng.integers(1, 6)))]
            mask = eval_tree(cols, tree)
            cnt = int(mask.sum())
            limit = int(rng.choice([0, 0, 1, 7, 33, cnt // 2 + 1, cnt, cnt + 1, nrows + 5]))
            for encoded in (False, True):
                what = f"seed {seed} q{qi} rows {nrows} block {block} x{seg_blocks} {'PFOR' if pfor else 'DENSE'} {env} flags {flags} enc {encoded}"
                st = refusal(terms, cols, proj, encoded, pfor, block, min(block, nrows))
                if st is None:
                    run(eng, "t", cols, tree, proj, limit, what, mask, encoded=encoded)
                    ran += 1
                else:
                    with pytest.raises(Imm3Error) as e:
                        eng.execute(Query("t", tree, Project(proj, limit)), real_or=True, encoded_filter=encoded)
                    assert e.value.status == st, (what, tree, proj, e.value)
                    refused += 1
    print(f"seed {seed}: {nrows} rows, blocks of {block}, {'PFOR' if pfor else 'DENSE'} id, {env} {flags}: {ran} ran, {refused} refused")


# ---- across ranks (device exchange) --------------------------------------------------------------------------------------

def _worker(rank, world, data_dir, port, out_dir):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch.distributed as dist

    import oracle_lib as O
    from immutable3_b200 import EQ, GT, LT, And, Engine, Match, Or, Project, Query, SegmentManager, Select
    from select_tree_ref import canonical_columns, eval_tree, expected_rows

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    os.environ["IMM3_PREFIX_ROWS"] = "8192"
    os.environ["IMM3_COMM_TIMEOUT_MS"] = "10000"
    try:
        with SegmentManager(data_dir, device=0, rank=rank, world=world) as sm, O.Oracle(data_dir) as whole:
            sm.comm_connect()
            eng = Engine(sm)
            cols = canonical_columns(whole, "t", ["id", "state", "age", "score"])
            ids = np.sort(cols["id"].astype(np.int64))
            q = lambda f: int(ids[int(f * (len(ids) - 1))])
            sels = [Or(Select("age", LT(5)), Select("age", GT(95))),
                    Or(And(Select("id", GT(q(0.1))), Select("id", LT(q(0.3)))), Select("state", Match(["CA"]))),
                    Or(Select("id", EQ(q(0.0))), Select("id", EQ(q(1.0)))),                               # the first and the last row
                    Or(And(Select("id", GT(q(0.8))), Select("age", LT(50))), Or(Select("age", EQ(7)), Select("score", LT(-990)))),
                    Or(Select("score", GT(5000)), Select("state", Match(["ZZ"])))]                       # nothing anywhere
            for sel in sels:
                mask = eval_tree(cols, sel)
                for proj in (["id"], ["id", "age", "state"]):
                    full = expected_rows(cols, mask, proj)
                    with eng.begin(Query("t", sel, Project(proj, 0)), real_or=True) as h:
                        c0 = h.rank_counts[0]
                    limits = [0, 1, 33, 5000] + [c for c in (c0 - 1, c0, c0 + 1) if c > 0]          # cuts at rank 0's count
                    for limit in limits:
                        want = [c[:limit] for c in full] if limit else full
                        with eng.begin(Query("t", sel, Project(proj, limit)), real_or=True) as h:
                            r = h.route
                            assert h.kernel_launches == (len(r.split(";")) if r else 0), (rank, sel, limit, r, h.kernel_launches)
                            assert h.global_count == len(want[0]), (rank, sel, limit, h.global_count, len(want[0]), h.route)
                            h.fetch(h.take)
                            for c in range(len(proj)):
                                got = h.column(c)
                                assert np.array_equal(got, want[c][h.global_offset:h.global_offset + h.take]), (rank, sel, limit, proj[c], h.route)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world, nrows", [(2, 30_000), (3, 30_000), (4, 5_000)])          # (5000 rows: two segments, empty slices)
def test_sharded(tmp_path, world, nrows):
    import torch.multiprocessing as mp

    data = tmp_path / "data"
    rng = np.random.default_rng(world)
    make_table(data, "t", nrows, 1024, 3, seed=4, id_mode="random", extra_cols=[("score:DENSE_INT", rng.integers(-1000, 1000, nrows).astype(np.int32))])
    port = 48300 + (os.getpid() % 1500) + 7 * world
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


# ---- 40 M rows: the default prefix size --------------------------------------------------------------------------------

def test_40m_rows_prefix_phases(tmp_path_factory):
    """LIMIT 10 and 1000 on 40 M rows take the prefix phase (4 M rows by default): rows early in it, rows only behind it, no
    rows; against numpy on the files."""
    d = tmp_path_factory.mktemp("or40m_prefix")
    n = 40_000_000
    O.synth_write(d, "syn", n)
    order = sorted(range(40), key=lambda i: f"id_{i}.dat")                # canonical order: 0, 1, 10, 11, ..., 19, 2, 20, ..., 9
    age_ = np.concatenate([np.fromfile(d / "syn" / f"age_{i}.dat", np.int8) for i in order])
    ids = np.concatenate([np.fromfile(d / "syn" / f"id_{i}.dat", "<i4") for i in order])
    st = np.concatenate([np.fromfile(d / "syn" / f"state_{i}.dat", "S2") for i in order])
    per = 1024 * 1000 + 1
    s9 = 9 * per                                                          # segment 9: the last in canonical order
    cases = [("early", Or(And(Select("age", GT(18)), Select("age", LT(30))), Select("id", LT(1000))), ((age_ > 18) & (age_ < 30)) | (ids < 1000)),
             ("late", Or(And(Select("id", GT(s9 + 100)), Select("id", LT(s9 + 5000))),
                         And(Select("id", GT(s9 + 20_000)), And(Select("id", LT(s9 + 900_000)), Select("state", Match(["CA"]))))),
              ((ids > s9 + 100) & (ids < s9 + 5000)) | ((ids > s9 + 20_000) & (ids < s9 + 900_000) & (st == b"CA"))),
             ("none", Or(Select("id", LT(-5)), Select("state", Match(["ZZ"]))), np.zeros(n, bool))]
    with SegmentManager(d) as sm:
        eng = Engine(sm)
        for key, sel, keep in cases:
            idx = np.flatnonzero(keep)
            if key == "late":
                assert idx[0] > 8 << 20
            for limit in (10, 1000):
                with eng.execute(Query("syn", sel, Project(["id", "age"], limit)), real_or=True) as got:
                    r = got.route
                    assert got.kernel_launches == len(r.split(";")), r
                    fa, fb = phases(r)
                    assert fa == 2 and fb == (0 if key == "early" else 2), (key, limit, r)
                    assert got.nrows == min(limit, len(idx)), (key, limit, got.nrows, r)
                    assert np.array_equal(got.column(0), ids[idx[:limit]]) and np.array_equal(got.column(1), age_[idx[:limit]]), (key, limit, r)
