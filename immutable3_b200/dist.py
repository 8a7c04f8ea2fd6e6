"""Segment-sharded execution: one process (rank) per GPU, contiguous canonical segment slices
(SURVEY.md §8e).  The data path has no collective: every rank scans its own slice.  The only
exchange is one int64 per rank — its local match count (already capped at LIMIT).  On GPUs the
library does it itself, on the device (peer stores over NVLink behind the query's last kernel,
`SegmentManager.comm_connect`, include/imm3.h imm3_comm_*); without a connected communicator (the
gloo CPU tests, which exercise the host arithmetic) it is a `torch.distributed.all_gather`.  Either
way each rank then knows its global output offset and how many of its leading rows survive the LIMIT cut.
Aggregates (`execute_agg`) exchange the partial groups themselves: merged on the GPUs on a connected handle
(imm3_query_agg_global), otherwise all-gathered and merged on the host in rank order (`merge_partials`).

The local executor is any object with `begin(query) -> handle` (handle.local_count) and
`finish(handle, take) -> list of numpy columns`.  The product executor is `CudaExecutor`
(immutable3_b200.engine.Engine over the C ABI).  Tests inject other executors to exercise the
offset/LIMIT arithmetic without GPUs; nothing in this module computes query results itself.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _lib as L
from .engine import Avg, Count, Engine, Max, Min, ProjectAgg, Query, Result, Sum


def shard_range(nsegments: int, rank: int, world: int):
    """Canonical slice [rank*n/world, (rank+1)*n/world) — same arithmetic as the C library."""
    return rank * nsegments // world, (rank + 1) * nsegments // world


def limit_split(counts: Sequence[int], limit: int):
    """(offsets, takes): exclusive scan of the per-rank counts and the rows each rank emits so that
    the concatenation in rank order is the first `limit` rows of the global canonical order
    (limit <= 0: unlimited; Project.scala:73-77)."""
    offsets, takes, run = [], [], 0
    for c in counts:
        offsets.append(run)
        takes.append(c if limit <= 0 else max(0, min(c, limit - run)))
        run += c
    return offsets, takes


def merge_partials(parts: Sequence[List[np.ndarray]], ngroup: int, aggs: Sequence) -> List[np.ndarray]:
    """The fan-in of ProjectAggregateQueueOp (ProjectAggregateQueue.scala:21-45) over per-rank partial groups, in rank
    order: `parts[r]` = rank r's columns (group columns, then one per aggregate).  A key takes the position of the first
    rank that holds it (global first-appearance order = rank order, then the rank's own order); Count and Sum add up
    (exactly: Python ints), Min / Max take the extreme.  The host form of what imm3_query_agg_global does on the GPUs.
    Avg does not merge: `sum_avg_partials` restates it as a Sum and a Count first."""
    pos, rows, firsts = {}, [], []
    for cols in parts:
        n = len(cols[0]) if cols else 0
        for i in range(n):
            key = tuple(cols[g][i].item() for g in range(ngroup))
            vals = [cols[ngroup + a][i].item() for a in range(len(aggs))]
            j = pos.get(key)
            if j is None:
                pos[key] = len(rows)
                rows.append(vals)
                firsts.append((cols, i))
                continue
            m = rows[j]
            for a, agg in enumerate(aggs):
                if isinstance(agg, (Count, Sum)):
                    m[a] += vals[a]
                elif isinstance(agg, Min):
                    m[a] = min(m[a], vals[a])
                elif isinstance(agg, Max):
                    m[a] = max(m[a], vals[a])
                else:
                    raise TypeError(f"not a mergeable aggregate: {agg!r}")
    template = next((cols for cols in parts if cols), None)
    if template is None:
        return []
    out = [np.array([c[g][i] for c, i in firsts], dtype=template[g].dtype) for g in range(ngroup)]
    out += [np.array([m[a] for m in rows], dtype=template[ngroup + a].dtype) for a in range(len(aggs))]
    return out


def sum_avg_partials(aggs: Sequence):
    """The aggregates a rank computes for a Sum / Avg query merged on the host: every Avg(c) becomes Sum(c), and one Count
    of the group's rows is carried (the query's first Count, else one appended).  Returns (those aggregates, the index of
    the Count)."""
    plan = [Sum(a.col, a.alias) if isinstance(a, Avg) else a for a in aggs]
    count = next((i for i, a in enumerate(plan) if isinstance(a, Count)), None)
    if count is None:
        plan.append(Count(aggs[0].col))
        count = len(plan) - 1
    return plan, count


def finish_sum_avg(cols: List[np.ndarray], ngroup: int, aggs: Sequence, count: int) -> List[np.ndarray]:
    """Merged columns of the `sum_avg_partials` plan -> the query's columns: Avg = float64(sum) / float64(count) (bitwise
    what imm3_query_agg_ext computes), the carried Count dropped unless the query asked for it.  A group of more than 2^32
    rows is refused as the library refuses it (its sum may not fit int64)."""
    if not cols:
        return []
    n = cols[ngroup + count]
    if len(n) and int(n.max()) > 1 << 32:
        raise L.Imm3Error(L.ERR_UNSUPPORTED, "a group of more than 2^32 rows: sum / avg are exact for groups of at most 2^32 rows")
    out = list(cols[:ngroup])
    for a, agg in enumerate(aggs):
        c = cols[ngroup + a]
        out.append(c.astype(np.float64) / n.astype(np.float64) if isinstance(agg, Avg) else c)
    return out


class CudaExecutor:
    def __init__(self, engine: Engine):
        self.engine = engine

    def begin(self, query: Query, sum_avg: bool = False, encoded_filter: bool = False) -> Result:
        if sum_avg or encoded_filter:
            return self.engine.begin(query, sum_avg=sum_avg, encoded_filter=encoded_filter)
        return self.engine.begin(query)

    def finish(self, handle: Result, take: int) -> List[np.ndarray]:
        handle.fetch(take)
        return handle.columns()


@dataclass
class ShardResult:
    rank: int
    world: int
    counts: List[int]      # local counts of every rank (each capped at LIMIT)
    offset: int            # global ordinal of this rank's first emitted row
    take: int              # rows this rank emits
    total: int             # rows of the whole result
    columns: List[np.ndarray]
    device_ms: float = 0.0


class ShardedEngine:
    def __init__(self, executor, group=None, collective_device: Optional[str] = None):
        import torch.distributed as dist

        self.executor = executor
        self.group = group
        self.dist = dist
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        if collective_device is None:
            collective_device = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        self.collective_device = collective_device

    def execute(self, query: Query) -> ShardResult:
        import torch

        h = self.executor.begin(query)
        if getattr(getattr(self.executor, "engine", None), "sm", None) is not None and self.executor.engine.sm.comm_connected:
            # the GPUs exchanged the counts themselves (imm3_comm_*): nothing to gather here
            counts = h.rank_counts
            cols = self.executor.finish(h, h.take)
            return ShardResult(self.rank, self.world, counts, h.global_offset, h.take, h.global_count, cols, float(h.device_ms))
        mine = torch.tensor([int(h.local_count)], dtype=torch.int64, device=self.collective_device)
        everyone = [torch.zeros_like(mine) for _ in range(self.world)]
        self.dist.all_gather(everyone, mine, group=self.group)  # the only exchange on the path
        counts = [int(t.item()) for t in everyone]
        offsets, takes = limit_split(counts, int(query.project.limit))
        cols = self.executor.finish(h, takes[self.rank])
        ms = float(getattr(h, "device_ms", 0.0))
        return ShardResult(self.rank, self.world, counts, offsets[self.rank], takes[self.rank], sum(takes), cols, ms)

    def execute_agg(self, query: Query, sum_avg: bool = False, encoded_filter: bool = False) -> ShardResult:
        """A ProjectAgg query over the whole table, the same groups on every rank: `columns` = the global groups,
        `counts` = every rank's partial group count, offset 0, take = total = the number of global groups.  On a
        connected handle the GPUs merge the partials themselves (imm3_query_agg_global); otherwise every rank's partial
        columns are all-gathered through torch.distributed and merged on the host in rank order (`merge_partials`).
        `sum_avg=True` resolves Sum / Avg (imm3_query_agg_ext; on the host path each rank computes Avg as a Sum and a
        Count, `sum_avg_partials`, and the merged sums are divided once, `finish_sum_avg`).  `encoded_filter=True` accepts
        predicates on sorted-int-codec columns (IMM3_AGG_ENCODED_FILTER, on the GPU merge and on every rank's partial query of
        the host merge alike)."""
        engine = getattr(self.executor, "engine", None)
        if getattr(getattr(engine, "sm", None), "comm_connected", False):
            with engine.execute_agg_global(query, sum_avg=sum_avg, encoded_filter=encoded_filter) as h:
                cols = h.columns()
                return ShardResult(self.rank, self.world, h.rank_counts, 0, h.nrows, h.nrows, cols, float(h.device_ms))
        aggs, ngroup = list(query.project.aggs), len(query.project.groupBy)
        kw = {"encoded_filter": True} if encoded_filter else {}
        if sum_avg:
            plan, count = sum_avg_partials(aggs)
            h = self.executor.begin(Query(query.table, query.select, ProjectAgg(plan, query.project.groupBy)), sum_avg=True, **kw)
        else:
            h = self.executor.begin(query, **kw)  # this rank's partial groups
        mine = self.executor.finish(h, int(h.local_count))
        everyone = [None] * self.world
        self.dist.all_gather_object(everyone, mine, group=self.group)
        if sum_avg:
            cols = finish_sum_avg(merge_partials(everyone, ngroup, plan), ngroup, aggs, count)
        else:
            cols = merge_partials(everyone, ngroup, aggs)
        total = len(cols[0]) if cols else 0
        counts = [len(p[0]) if p else 0 for p in everyone]
        return ShardResult(self.rank, self.world, counts, 0, total, total, cols, float(getattr(h, "device_ms", 0.0)))

    def gather_rows(self, res: ShardResult, dst: int = 0):
        """Concatenate every rank's emitted rows on `dst` in rank order (= canonical order). Test helper."""
        payload = [c for c in res.columns]
        gathered = [None] * self.world if self.rank == dst else None
        self.dist.gather_object(payload, gathered, dst=dst, group=self.group)
        if self.rank != dst:
            return None
        ncols = len(payload)
        return [np.concatenate([g[c] for g in gathered]) for c in range(ncols)]
