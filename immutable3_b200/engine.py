"""Host-side mirror of the reference's Table / SegmentManager / Query / Engine interface.

Same names and argument meaning as the Scala (so the parity tests read like reference usage):

    sm = SegmentManager(data_dir)                       # SegmentManager.scala:20
    table = sm.getTable("test_100m")                    # SegmentManager.scala:89
    engine = Engine(sm)                                 # Engine.scala:81
    query = Query(table.name,
                  And(Select("age", GT(18)), Select("age", LT(30))),
                  Project(["id", "age"], 10))           # Query.scala:3-46
    for row in engine.execute(query): print(row)        # Engine.scala:158, SqlCli.scala:70-73

Everything here is thin: the ADT is flattened to the imm3_pred list of include/imm3.h and handed to
the CUDA library.  There is no compute and no fallback on this side.
"""
from __future__ import annotations

import ctypes as C
import weakref
from dataclasses import dataclass, field
from typing import Iterator, List, Optional, Sequence, Union

import numpy as np

from . import _lib as L

# ------------------------------------------------------------------------------------------------
# Query ADT (Query.scala:3-46)
# ------------------------------------------------------------------------------------------------


class SelectCondition:
    pass


@dataclass(frozen=True)
class Match(SelectCondition):
    values: Sequence[str]


@dataclass(frozen=True)
class NotMatch(SelectCondition):
    values: Sequence[str]


@dataclass(frozen=True)
class EQ(SelectCondition):
    eq: float


@dataclass(frozen=True)
class GT(SelectCondition):
    gt: float


@dataclass(frozen=True)
class LT(SelectCondition):
    lt: float


class NoOp(SelectCondition):
    pass


class SelectADT:
    pass


@dataclass(frozen=True)
class And(SelectADT):
    op1: SelectADT
    op2: SelectADT


@dataclass(frozen=True)
class Or(SelectADT):
    op1: SelectADT
    op2: SelectADT


@dataclass(frozen=True)
class Select(SelectADT):
    col: str
    cond: SelectCondition


class _NoSelect(SelectADT):
    def __repr__(self):
        return "NoSelect"


NoSelect = _NoSelect()


@dataclass(frozen=True)
class Project:
    cols: Sequence[str]
    limit: int = 0


# Aggregates (Query.scala:17-27).  Sum / Avg exist in the ADT and the parser, but Engine.resolveProjectOp throws on them
# (Engine.scala:153): by default they come back as IMM3_ERR_UNSUPPORTED, as there.  `sum_avg=True` (Engine.execute,
# execute_agg_global, ShardedEngine.execute_agg) resolves them through imm3_query_agg_ext: Sum = the exact int64 sum,
# Avg = float64(sum) / float64(count).
# A predicate on a sorted-int-codec column in a ProjectAgg query is refused (IMM3_ERR_UNSUPPORTED) unless
# `encoded_filter=True` (the same methods), which sets IMM3_AGG_ENCODED_FILTER on imm3_query_agg_ext: the block filter
# kernels decide such predicates and the aggregation reads their per-block selection.  The two keywords are independent:
# `encoded_filter=True` alone still refuses Sum / Avg as the parity path does.
@dataclass(frozen=True)
class Sum:
    col: str
    alias: Optional[str] = None


@dataclass(frozen=True)
class Avg:
    col: str
    alias: Optional[str] = None


@dataclass(frozen=True)
class Min:
    col: str
    alias: Optional[str] = None


@dataclass(frozen=True)
class Max:
    col: str
    alias: Optional[str] = None


@dataclass(frozen=True)
class Count:
    col: str
    alias: Optional[str] = None


@dataclass(frozen=True)
class ProjectAgg:
    aggs: Sequence
    groupBy: Sequence[str] = ()


@dataclass(frozen=True)
class Query:
    table: str
    select: SelectADT
    project: Project


def flatten_select(sel: SelectADT) -> List[Select]:
    """Leaves of the select tree in the order PipelineThread.runOps applies them
    (Engine.scala:237-245: rec(n2)(rec(n1)(x)) — n1 first; the AND/OR tag is ignored, so `Or`
    is evaluated as a conjunction exactly like the reference, SURVEY.md §3.4-7)."""
    if isinstance(sel, (And, Or)):
        return flatten_select(sel.op1) + flatten_select(sel.op2)
    if isinstance(sel, Select):
        return [sel]
    if sel is NoSelect or isinstance(sel, _NoSelect):
        return []
    raise TypeError(f"not a SelectADT: {sel!r}")


MAX_OR_TERMS = 16  # IMM3_MAX_OR_TERMS


def select_dnf(sel: SelectADT) -> List[List[Select]]:
    """The select tree in disjunctive normal form - what `a or b` MEANS, as opposed to what the reference does with it
    (flatten_select above).  A list of conjunctions, each a list of leaves in application order; [[]] = no predicate.
    And distributes over Or: And(Or(a, b), c) -> [[a, c], [b, c]]."""
    if isinstance(sel, Or):
        terms = select_dnf(sel.op1) + select_dnf(sel.op2)
    elif isinstance(sel, And):
        terms = [l + r for l in select_dnf(sel.op1) for r in select_dnf(sel.op2)]
    elif isinstance(sel, Select):
        terms = [[sel]]
    elif sel is NoSelect or isinstance(sel, _NoSelect):
        terms = [[]]
    else:
        raise TypeError(f"not a SelectADT: {sel!r}")
    if len(terms) > MAX_OR_TERMS:
        raise L.Imm3Error(L.ERR_UNSUPPORTED, f"the select tree expands to {len(terms)} conjunctions (at most {MAX_OR_TERMS})")
    return terms


def _pred_array(leaves: Sequence[Select]):
    """imm3_pred[] + the ctypes objects that must stay alive while it is used."""
    n = len(leaves)
    arr = (L.Pred * max(1, n))()
    keep = []
    for i, leaf in enumerate(leaves):
        arr[i].col = leaf.col.encode()
        c = leaf.cond
        if isinstance(c, GT):
            arr[i].op, arr[i].num = L.OP_GT, float(c.gt)
        elif isinstance(c, LT):
            arr[i].op, arr[i].num = L.OP_LT, float(c.lt)
        elif isinstance(c, EQ):
            arr[i].op, arr[i].num = L.OP_EQ, float(c.eq)
        elif isinstance(c, (Match, NotMatch)):
            arr[i].op = L.OP_MATCH if isinstance(c, Match) else L.OP_NOTMATCH
            strs = L.cstr_array(list(c.values))
            keep.append(strs)
            arr[i].strs = C.cast(strs, C.POINTER(C.c_char_p))
            arr[i].nstrs = len(c.values)
        else:
            arr[i].op = L.OP_NOOP
    return arr, n, keep


# ------------------------------------------------------------------------------------------------
# Row / result (Record.scala:3-14, Project.scala:17-81)
# ------------------------------------------------------------------------------------------------


class Row(tuple):
    def __repr__(self):  # Row.toString: xs.mkString("Row(", ",", ")")
        return "Row(" + ",".join(str(x) for x in self) + ")"

    __str__ = __repr__


_NP = {L.COL_INT: np.dtype("<i4"), L.COL_TINYINT: np.dtype("i1"), L.COL_COUNT: np.dtype("<i8"), L.COL_DOUBLE: np.dtype("<f8"),
       L.COL_INT64: np.dtype("<i8")}
_AGG_OPS = {"Count": L.AGG_COUNT, "Min": L.AGG_MIN, "Max": L.AGG_MAX, "Sum": L.AGG_SUM, "Avg": L.AGG_AVG}


class Result:
    """Rows of one query in canonical order, column-major (owns an imm3_result)."""

    def __init__(self, handle: int, lib, sm=None):
        self._h = handle
        self._lib = lib
        self._sm = sm  # keeps the SegmentManager (and its imm3_db) alive for as long as this result is open
        if sm is not None:
            sm._results.add(self)

    # -- two-phase API (sharded execution) --
    @property
    def local_count(self) -> int:
        return int(self._lib.imm3_result_local_count(self._h))

    # -- placement in the global result after the on-device count exchange (single handle: 0 / all / all) --
    @property
    def global_offset(self) -> int:
        return int(self._lib.imm3_result_global_offset(self._h))

    @property
    def take(self) -> int:
        return int(self._lib.imm3_result_take(self._h))

    @property
    def global_count(self) -> int:
        return int(self._lib.imm3_result_global_count(self._h))

    @property
    def rank_counts(self) -> List[int]:
        buf = (C.c_int64 * 16)()
        n = L.check(self._lib.imm3_result_rank_counts(self._h, buf, 16))
        return [int(buf[i]) for i in range(n)]

    def fetch(self, nrows: int) -> "Result":
        L.check(self._lib.imm3_result_fetch(self._h, int(nrows)))
        return self

    def fetch_async(self, nrows: int) -> "Result":
        """Queue the device->host copies of the first `nrows` rows and return; `wait()` makes them readable."""
        L.check(self._lib.imm3_result_fetch_async(self._h, int(nrows)))
        return self

    def wait(self) -> "Result":
        L.check(self._lib.imm3_result_wait(self._h))
        return self

    # -- accessors --
    @property
    def nrows(self) -> int:
        return int(self._lib.imm3_result_nrows(self._h))

    @property
    def ncols(self) -> int:
        return int(self._lib.imm3_result_ncols(self._h))

    @property
    def device_ms(self) -> float:
        return float(self._lib.imm3_result_device_ms(self._h))

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.imm3_result_kernel_launches(self._h))

    @property
    def route(self) -> str:
        """The kernels the query queued, in launch order: "blocks_prune;blocks_filter_lane/w=11/s=2;blocks_group_emit/ctas=148"."""
        return (self._lib.imm3_result_route(self._h) or b"").decode()

    def stage_ms(self, stage: int) -> float:
        return float(self._lib.imm3_result_stage_ms(self._h, stage))

    def host_us(self):
        """Wall clock inside imm3_query_begin by phase: [plan, buffers + device plan, launches, wait for the GPU, epilogue]."""
        return [float(self._lib.imm3_result_host_us(self._h, i)) for i in range(5)]

    @property
    def algorithmic_bytes(self) -> int:
        return int(self._lib.imm3_result_algorithmic_bytes(self._h))

    def col_name(self, c: int) -> str:
        return self._lib.imm3_result_col_name(self._h, c).decode()

    def col_type(self, c: int) -> int:
        return int(self._lib.imm3_result_col_type(self._h, c))

    def col_width(self, c: int) -> int:
        return int(self._lib.imm3_result_col_width(self._h, c))

    def column(self, c: int) -> np.ndarray:
        """Copy of column c: int32 / int8 array, or an S<k> bytes array for STRING(k)."""
        n, w, t = self.nrows, self.col_width(c), self.col_type(c)
        dt = _NP.get(t, np.dtype(f"S{w}"))
        if n == 0:
            return np.empty(0, dtype=dt)
        ptr = self._lib.imm3_result_col_data(self._h, c)
        raw = (C.c_uint8 * (n * w)).from_address(ptr)
        return np.frombuffer(raw, dtype=dt, count=n).copy()

    def columns(self) -> List[np.ndarray]:
        return [self.column(c) for c in range(self.ncols)]

    def format_row(self, i: int) -> str:
        buf = C.create_string_buffer(4096)
        L.check(self._lib.imm3_result_format_row(self._h, i, buf, len(buf)))
        return buf.value.decode("utf-8", "replace")

    def __iter__(self) -> Iterator[Row]:
        cols = self.columns()
        types = [self.col_type(c) for c in range(self.ncols)]
        for i in range(self.nrows):
            yield Row(
                cols[c][i].decode("utf-8", "replace") if types[c] == L.COL_STRING else (float(cols[c][i]) if types[c] == L.COL_DOUBLE else int(cols[c][i]))
                for c in range(len(cols))
            )

    def __len__(self):
        return self.nrows

    def close(self):
        if self._h:
            self._lib.imm3_result_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


# ------------------------------------------------------------------------------------------------
# Table / Column / SegmentManager (Table.scala:9, Column.scala:18, SegmentManager.scala:20-112)
# ------------------------------------------------------------------------------------------------


@dataclass(frozen=True)
class Column:
    name: str
    columnType: str  # "INT" | "TINYINT" | "STRING"
    codec: str       # "PFOR_INT" | "DENSE_INT" | "DENSE_TINYINT" | "DENSE_STRING"
    width: int
    encoded_bytes: int = 0


@dataclass(frozen=True)
class Table:
    name: str
    columns: Sequence[Column]
    blockSize: int
    nsegments: int = 0
    seg_begin: int = 0
    seg_end: int = 0
    nrows: int = 0
    nblocks: int = 0
    resident_bytes: int = 0

    def getColumn(self, colName: str) -> Column:
        for c in self.columns:
            if c.name == colName:
                return c
        raise KeyError(f"Column {colName} does not exist in table {self.name}")


_CT = ["INT", "TINYINT", "STRING"]
_CODEC = ["PFOR_INT", "DENSE_INT", "DENSE_TINYINT", "DENSE_STRING"]


class SegmentManager:
    """`new SegmentManager(dataDir)`: discovers every table under data_dir and stages this
    handle's canonical segment slice into HBM (imm3_open)."""

    def __init__(self, dataDir: str, device: int = 0, rank: int = 0, world: int = 1, flags: int = 0):
        self._lib = L.lib()
        self._h = C.c_void_p()
        opts = L.OpenOpts(device, rank, world, flags)
        self._results = weakref.WeakSet()  # open results of this handle: closed before the handle is
        self.comm_connected = False
        L.check(self._lib.imm3_open(str(dataDir).encode(), C.byref(opts), C.byref(self._h)))
        self.dataDir = str(dataDir)
        self.rank, self.world, self.flags = rank, world, flags

    def comm_connect(self, group=None) -> "SegmentManager":
        """Connect the ranks' count mailboxes (imm3_comm_*): after this, every query exchanges the per-rank match counts
        on the GPUs over NVLink.  The 64-byte IPC handles travel once through torch.distributed (bootstrap only)."""
        if self.world == 1:
            return self
        import torch.distributed as dist

        mine = (C.c_uint8 * L.COMM_HANDLE_BYTES)()
        L.check(self._lib.imm3_comm_local_handle(self._h, mine))
        everyone = [None] * self.world
        dist.all_gather_object(everyone, bytes(mine), group=group)
        blob = C.create_string_buffer(b"".join(everyone), self.world * L.COMM_HANDLE_BYTES)
        L.check(self._lib.imm3_comm_connect(self._h, blob, self.world))
        self.comm_connected = True
        dist.barrier(group=group)  # nobody queries before every rank has mapped every mailbox
        return self

    @property
    def handle(self):
        return self._h

    @property
    def tables(self) -> List[Table]:
        n = self._lib.imm3_table_count(self._h)
        return [self.getTable(self._lib.imm3_table_name(self._h, i).decode()) for i in range(n)]

    def getTable(self, tableName: str) -> Table:
        d = L.TableDesc()
        L.check(self._lib.imm3_table_info(self._h, tableName.encode(), C.byref(d)))
        cols = []
        for i in range(d.ncols):
            cd = L.ColumnDesc()
            L.check(self._lib.imm3_column_info(self._h, tableName.encode(), i, C.byref(cd)))
            cols.append(Column(cd.name.decode(), _CT[cd.column_type], _CODEC[cd.codec], cd.width, cd.encoded_bytes))
        return Table(tableName, cols, d.block_size, d.nsegments, d.seg_begin, d.seg_end, d.nrows, d.nblocks, d.resident_bytes)

    def getTableSegmentCount(self, tableName: str) -> int:
        return self.getTable(tableName).nsegments

    def segmentFileIds(self, tableName: str) -> List[int]:
        """Numeric ids of the segment files in canonical (file-name-sorted) order."""
        out = []
        v = C.c_int32()
        for i in range(self.getTableSegmentCount(tableName)):
            L.check(self._lib.imm3_segment_file_id(self._h, tableName.encode(), i, C.byref(v)))
            out.append(v.value)
        return out

    def reupload(self, tableName: str, cols: Optional[Sequence[str]] = None) -> int:
        n = C.c_int64()
        if cols:
            arr = L.cstr_array(list(cols))
            L.check(self._lib.imm3_reupload(self._h, tableName.encode(), C.cast(arr, C.POINTER(C.c_char_p)), len(cols), C.byref(n)))
        else:
            L.check(self._lib.imm3_reupload(self._h, tableName.encode(), None, 0, C.byref(n)))
        return n.value

    def set_stream(self, cuda_stream: int):
        L.check(self._lib.imm3_set_stream(self._h, C.c_void_p(cuda_stream)))

    def sync(self):
        L.check(self._lib.imm3_sync(self._h))

    def close(self):
        if self._h:
            for r in list(self._results):
                r.close()
            L.check(self._lib.imm3_close(self._h))
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


# ------------------------------------------------------------------------------------------------
# Engine (Engine.scala:81-232, Project branch)
# ------------------------------------------------------------------------------------------------


class Engine:
    def __init__(self, sm: SegmentManager):
        self.sm = sm
        self._lib = sm._lib

    def _call(self, fn, query: Query):
        if not isinstance(query.project, Project):
            raise L.Imm3Error(L.ERR_UNSUPPORTED, "only Project queries are on the scan/filter/project path")
        preds, npreds, keep = _pred_array(flatten_select(query.select))
        proj = L.cstr_array(list(query.project.cols))
        out = C.c_void_p()
        L.check(fn(self.sm.handle, query.table.encode(), preds, npreds, C.cast(proj, C.POINTER(C.c_char_p)),
                   len(query.project.cols), int(query.project.limit), C.byref(out)))
        del keep
        return Result(out, self._lib, self.sm)

    def prepare(self, query: Query):
        """The argument marshalling of `begin`, done once: `begin_prepared(p)` then costs one foreign call per query (a
        caller that repeats a query - the benchmark, a dashboard - keeps Python out of the measured path)."""
        if not isinstance(query.project, Project):
            raise L.Imm3Error(L.ERR_UNSUPPORTED, "only Project queries are on the scan/filter/project path")
        preds, npreds, keep = _pred_array(flatten_select(query.select))
        proj = L.cstr_array(list(query.project.cols))
        return (query.table.encode(), preds, npreds, C.cast(proj, C.POINTER(C.c_char_p)), len(query.project.cols),
                int(query.project.limit), (keep, proj))

    def begin_prepared(self, p) -> Result:
        out = C.c_void_p()
        L.check(self._lib.imm3_query_begin(self.sm.handle, p[0], p[1], p[2], p[3], p[4], p[5], C.byref(out)))
        return Result(out, self._lib, self.sm)

    def execute(self, query: Query, real_or: bool = False, sum_avg: bool = False, encoded_filter: bool = False) -> Result:
        """Engine.execute: the rows of the query in canonical order (iterate for Row objects).  `real_or=True` evaluates
        Or as a disjunction (imm3_query_begin_dnf) instead of the reference's Or == And (Engine.scala:236-245).
        `sum_avg=True` resolves Sum / Avg in a ProjectAgg query (imm3_query_agg_ext), which the reference refuses.
        `encoded_filter=True` accepts predicates on sorted-int-codec columns in a ProjectAgg query (IMM3_AGG_ENCODED_FILTER),
        and with `real_or=True` in the terms of a disjunction (imm3_query_begin_dnf_ext, IMM3_DNF_ENCODED_FILTER)."""
        if isinstance(query.project, ProjectAgg):
            return self._call_agg(query, sum_avg=sum_avg, encoded_filter=encoded_filter)
        if real_or:
            r = self.begin(query, real_or=True, encoded_filter=encoded_filter)
            return r.fetch(r.take)
        return self._call(self._lib.imm3_query, query)

    def begin(self, query: Query, real_or: bool = False, sum_avg: bool = False, encoded_filter: bool = False) -> Result:
        """First phase of a sharded query: kernels done, local match count known, nothing fetched."""
        if isinstance(query.project, ProjectAgg):
            return self._call_agg(query, sum_avg=sum_avg, encoded_filter=encoded_filter)
        if real_or:
            return self._call_dnf(query, encoded_filter)
        return self._call(self._lib.imm3_query_begin, query)

    def _call_dnf(self, query: Query, encoded_filter: bool = False) -> Result:
        if not isinstance(query.project, Project):
            raise L.Imm3Error(L.ERR_UNSUPPORTED, "only Project queries are on the scan/filter/project path")
        terms = select_dnf(query.select)
        preds, _, keep = _pred_array([leaf for t in terms for leaf in t])
        sizes = (C.c_int32 * len(terms))(*[len(t) for t in terms])
        proj = L.cstr_array(list(query.project.cols))
        out = C.c_void_p()
        args = (self.sm.handle, query.table.encode(), preds, sizes, len(terms), C.cast(proj, C.POINTER(C.c_char_p)), len(query.project.cols),
                int(query.project.limit))
        if encoded_filter:
            L.check(self._lib.imm3_query_begin_dnf_ext(*args, L.DNF_FLAG_ENCODED_FILTER, C.byref(out)))
        else:
            L.check(self._lib.imm3_query_begin_dnf(*args, C.byref(out)))
        del keep
        return Result(out, self._lib, self.sm)

    def execute_agg_global(self, query: Query, sum_avg: bool = False, encoded_filter: bool = False) -> Result:
        """A ProjectAgg query over the WHOLE table on every rank of a sharded handle (imm3_query_agg_global): the ranks'
        partial groups are merged on the GPUs over the communicator (`SegmentManager.comm_connect`).  On a single handle the
        result is that of `execute`; an unconnected sharded handle raises (IMM3_ERR_STATE).  `sum_avg` and
        `encoded_filter` as in `execute`."""
        return self._call_agg(query, glob=True, sum_avg=sum_avg, encoded_filter=encoded_filter)

    def _call_agg(self, query: Query, glob: bool = False, sum_avg: bool = False, encoded_filter: bool = False) -> Result:
        """Engine.execute, ProjectAgg branch (Engine.scala:200-232): one row per group, group columns then aggregates."""
        if not isinstance(query.project, ProjectAgg):
            raise L.Imm3Error(L.ERR_UNSUPPORTED, "not a ProjectAgg query")
        preds, npreds, keep = _pred_array(flatten_select(query.select))
        aggs = list(query.project.aggs)
        arr = (L.Agg * max(1, len(aggs)))()
        for i, a in enumerate(aggs):
            arr[i].col = a.col.encode()
            arr[i].op = _AGG_OPS[type(a).__name__]
        groups = L.cstr_array(list(query.project.groupBy))
        out = C.c_void_p()
        args = (self.sm.handle, query.table.encode(), preds, npreds, arr, len(aggs), C.cast(groups, C.POINTER(C.c_char_p)), len(query.project.groupBy))
        if encoded_filter and not sum_avg and any(isinstance(a, (Sum, Avg)) for a in aggs):
            # (imm3_query_agg_ext would resolve them: refuse them as the parity path does, so that the keywords stay independent)
            raise L.Imm3Error(L.ERR_UNSUPPORTED, "Unknown Aggregate type (Engine.scala:153: only Min, Max and Count are resolved)")
        if sum_avg or encoded_filter:
            flags = (L.AGG_FLAG_GLOBAL if glob else 0) | (L.AGG_FLAG_ENCODED_FILTER if encoded_filter else 0)
            L.check(self._lib.imm3_query_agg_ext(*args, flags, C.byref(out)))
        else:
            L.check((self._lib.imm3_query_agg_global if glob else self._lib.imm3_query_agg)(*args, C.byref(out)))
        del keep
        return Result(out, self._lib, self.sm)

    def execute_sql(self, sql: str) -> Result:
        """Same text as `SqlCli -q` (SQLParser.scala)."""
        out = C.c_void_p()
        L.check(self._lib.imm3_query_sql(self.sm.handle, sql.encode(), C.byref(out)))
        return Result(out, self._lib, self.sm)

    def filter_bitmap(self, table: str, select: SelectADT):
        """Selection bitmap of the conjunction (uint32 words, bit i of word w = canonical row 32w+i)."""
        preds, npreds, keep = _pred_array(flatten_select(select))
        words = C.POINTER(C.c_uint32)()
        nwords, nsel = C.c_int64(), C.c_int64()
        L.check(self._lib.imm3_filter_bitmap(self.sm.handle, table.encode(), preds, npreds, C.byref(words), C.byref(nwords), C.byref(nsel)))
        del keep
        arr = np.ctypeslib.as_array(words, shape=(max(1, nwords.value),))[: nwords.value].copy() if nwords.value else np.empty(0, np.uint32)
        return arr, nsel.value

    def explain(self, query: Query) -> dict:
        import json

        preds, npreds, keep = _pred_array(flatten_select(query.select))
        proj = L.cstr_array(list(query.project.cols))
        js = C.c_char_p()
        L.check(self._lib.imm3_explain(self.sm.handle, query.table.encode(), preds, npreds, C.cast(proj, C.POINTER(C.c_char_p)),
                                       len(query.project.cols), int(query.project.limit), C.byref(js)))
        del keep
        return json.loads(js.value.decode())
