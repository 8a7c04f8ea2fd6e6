#!/usr/bin/env python
"""bench.py — scan + filter + project throughput of the B200 path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|c3|...] [--rows R] [--scaling strong|weak]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # CPU restatement of the reference path on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's result rows to DIR/*.npy (dump_outputs)

Default = the north_star configuration (BASELINE.json configs[3], C4): the 1 B-row synthetic table with a
sorted-int-codec `id` column, `select id from test_1b where (id > L and id < H)` (1 % window), the canonical segment
list STRONG-sharded over the N GPUs (rows_total = 1e9 at every N; one contiguous slice per rank, SegmentManager.scala:41
order, one unit of work per segment as in Engine.scala:176-180).  A "step" is one query over the whole resident table.

Printed keys (one JSON line on rank 0):
  value        rows/s = rows_total / median over the K steps of [max over ranks of the WALL time from a host barrier to
               "every kernel of the query and the count exchange done, counts on the host" (imm3_query_begin returning)].
               The per-rank match counts are exchanged by the GPUs themselves over NVLink inside that span (imm3_comm_*).
  timing       the same steps' CUDA-event times (first kernel -> end of the exchange kernel), host overhead per query
  e2e          rows/s through the C ABI from PINNED HOST buffers: per step the query's columns are re-staged host->HBM,
               the query runs, and this rank's share of the result rows is copied to host memory
  e2e_resident the same with the table resident (SegmentManager loads once, Engine.execute per query)
  roofline     algorithmic bytes (SURVEY.md 8d) of one query / CUDA-event time of its kernels vs the measured HBM peak
  cpu_baseline the oracle (CPU restatement, kind "port") timed on this box's host cores on the same table (N=1 only)
  result_equal per rank: the fetched result columns are byte-identical (CRC-32 and length) to the oracle's over the slice
  workloads    secondary records measured the same way in the same run (C2 / C3 on test_100m, C5 points)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK, SEGMENT = 1024, 1000
ROWS_PER_SEG = BLOCK * SEGMENT + 1
METRIC = "rows/sec for scan+filter+project"

# name: (description, table kind)   kind "pfor" = test_1b schema (id:PFOR_INT), "dense" = test_100m schema (id:DENSE_INT)
WORKLOADS = {
    "c4": ("C4 test_1b (id:PFOR_INT sorted-int codec): select id from test_1b where (id > L and id < H), 1% window", "pfor"),
    "c4_limit10": ("C5 test_1b: select id from test_1b where (id > L and id < H) limit 10, 1% window", "pfor"),
    "c4dense": ("C4 dense-id twin: select id from t where (id > L and id < H), 1% window", "dense"),
    "c2": ("C2 test_100m: select id, age from test_100m where (age > 18 and age < 30)", "dense"),
    "c3": ("C3 test_100m: select id, state, age from test_100m where (state = 'CA' and age > 18 and age < 30)", "dense"),
    "c2p": ("C2 on test_1b (id:PFOR_INT): select id, age from test_1b where (age > 18 and age < 30)", "pfor"),
    "c5_rare": ("C5 test_1b: select id, state, age from test_1b where (state = 'CA' and age = 7)", "pfor"),
    "c5_rare_limit10": ("C5 test_1b: select id, state, age from test_1b where (state = 'CA' and age = 7) limit 10", "pfor"),
    "c5_limit10": ("C5 select id, age where (age > 18 and age < 30) limit 10", "dense"),
    "agg": ("Engine.scala:66-78 example: select min(age), max(age) from test_100m where age > 18 group by state", "dense"),
    "agg_count": ("select count(id), max(id) from test_100m where (age > 18 and age < 30) group by state, age", "dense"),
    "x_age": ("X select age where (age > 18 and age < 30)", "dense"),
    "x_id": ("X select id where (age > 18 and age < 30)", "dense"),
    "x_count": ("X select <nothing> where (age > 18 and age < 30)", "dense"),
    "x_none": ("X select id, age where age = 127 (no match)", "dense"),
    "x_all": ("X select id, age (no predicate)", "dense"),
    "x_1pct": ("X select id, age where age = 7", "dense"),
    **{f"x_lt{t}": (f"C5 scattered: select id, age where age < {t} ({t} %)", "dense") for t in (1, 2, 3, 4, 5, 6, 8, 10, 25, 50)},
    **{f"c5p_lt{t}": (f"C5 scattered on test_1b: select id, age where age < {t} ({t} %)", "pfor") for t in (1, 10, 50, 100)},
    **{f"c5p_lt{t}_limit10": (f"C5 scattered on test_1b: select id, age where age < {t} limit 10", "pfor") for t in (1, 10, 50, 100)},
    **{f"c5w_{n}": (f"C5 id window {p} of test_1b: select id where (id > L and id < H)", "pfor")
       for n, p in (("001", "0.01%"), ("01", "0.1%"), ("1", "1%"), ("10", "10%"), ("50", "50%"), ("100", "100%"))},
    **{f"c5w_{n}_limit10": (f"C5 id window {p} of test_1b: select id where (id > L and id < H) limit 10", "pfor")
       for n, p in (("001", "0.01%"), ("01", "0.1%"), ("1", "1%"), ("10", "10%"), ("50", "50%"), ("100", "100%"))},
}
# --sweep: BASELINE.json configs[4] (SURVEY.md 8d C5) - selectivity 0.01 % .. 100 % on test_1b, LIMIT 10 vs none, at N GPUs
SWEEP = [f"c5w_{n}" for n in ("001", "01", "1", "10", "50", "100")] + [f"c5p_lt{t}" for t in (1, 10, 50, 100)] + ["c5_rare"]
# what the default run measures besides the headline: (record name, workload, table rows)
AGG_SPECS = {  # workload -> (predicates, aggregates as (op, col) with op 0 = count, 1 = min, 2 = max, group-by columns)
    "agg": ([("age", 1, 18)], [(1, "age"), (2, "age")], ["state"]),
    "agg_count": ([("age", 1, 18), ("age", 2, 30)], [(0, "id"), (2, "id")], ["state", "age"]),
}
SECONDARY = [("c4_pruned_1b", "c4", None), ("agg_100m", "agg", 100_000_000), ("c2_100m", "c2", 100_000_000), ("c3_100m", "c3", 100_000_000), ("c4_limit10_1b", "c4_limit10", None),
             ("c5_rare_1b", "c5_rare", None), ("c5p_lt10_1b", "c5p_lt10", None)]
WINDOW_FRAC = {"c5w_001": 1e-4, "c5w_01": 1e-3, "c5w_1": 1e-2, "c5w_10": 0.1, "c5w_50": 0.5, "c5w_100": 1.0}
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much in all


def query_spec(workload: str, total_rows: int):
    """(predicates as (col, op, value), projection, limit) - plain data, shared by both arms."""
    GT, LT, EQ, MATCH = 1, 2, 3, 4
    age_range = [("age", GT, 18), ("age", LT, 30)]
    if workload in ("c4", "c4dense", "c4_limit10") or workload.replace("_limit10", "") in WINDOW_FRAC:
        frac = WINDOW_FRAC.get(workload.replace("_limit10", ""), 0.01)
        half = int(total_rows * frac / 2)
        lo, hi = total_rows // 2 - half, total_rows // 2 + half
        if frac >= 1.0:
            lo, hi = -1, total_rows
        return [("id", GT, lo), ("id", LT, hi)], ["id"], 10 if workload.endswith("limit10") else 0
    if workload in ("c2", "c2p"):
        return age_range, ["id", "age"], 0
    if workload == "c3":
        return [("state", MATCH, ["CA"])] + age_range, ["id", "state", "age"], 0
    if workload in ("c5_rare", "c5_rare_limit10"):
        return [("state", MATCH, ["CA"]), ("age", EQ, 7)], ["id", "state", "age"], 10 if workload.endswith("limit10") else 0
    if workload == "c5_limit10":
        return age_range, ["id", "age"], 10
    if workload.startswith("c5p_lt"):
        t = int(workload[6:].split("_")[0])
        return [("age", LT, t)], ["id", "age"], 10 if workload.endswith("limit10") else 0
    if workload.startswith("x_lt"):
        return [("age", LT, int(workload[4:]))], ["id", "age"], 0
    proj = {"x_age": ["age"], "x_id": ["id"], "x_count": []}.get(workload, ["id", "age"])
    preds = {"x_none": [("age", EQ, 127)], "x_all": [], "x_1pct": [("age", EQ, 7)]}.get(workload, age_range)
    return preds, proj, 0


def build_query(workload: str, table: str, total_rows: int):
    from immutable3_b200 import EQ, GT, LT, And, Count, Match, Max, Min, NoSelect, Project, ProjectAgg, Query, Select

    if workload in AGG_SPECS:
        preds, aggs, group_by = AGG_SPECS[workload]
        proj, limit = None, 0
    else:
        preds, proj, limit = query_spec(workload, total_rows)
    leaves = [Select(c, {1: GT, 2: LT, 3: EQ}[op](v)) if op != 4 else Select(c, Match(v)) for c, op, v in preds]
    sel = NoSelect
    for i, leaf in enumerate(leaves):
        sel = leaf if i == 0 else And(sel, leaf)
    if proj is None:
        return Query(table, sel, ProjectAgg([{0: Count, 1: Min, 2: Max}[op](col) for op, col in aggs], group_by))
    return Query(table, sel, Project(proj, limit))


def table_name(kind: str) -> str:
    return "test_1b" if kind == "pfor" else "test_100m"


def data_dir_for(kind: str, total_rows: int) -> str:
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
    return os.path.join(base, f"imm3_bench_{kind}_{total_rows}")


def nsegments(total_rows: int) -> int:
    return (total_rows + ROWS_PER_SEG - 1) // ROWS_PER_SEG


def ensure_table(kind: str, total_rows: int, rank: int, world: int, barrier, writer: str):
    """Write the synthetic table once (reused by later runs and by the other arm: both writers emit the same bytes,
    tests/test_writer_layout.py).  Rank 0 clears the directory and writes _table.meta, then every rank writes its share
    of the segment files.  writer = "product" (imm3_synth_write) or "oracle" (orc_synth_write; reference arm)."""
    d, table = data_dir_for(kind, total_rows), table_name(kind)
    done = os.path.join(d, table, ".complete_all")
    t0 = time.time()
    if os.path.exists(done):
        barrier()
        return d, table, 0.0
    nseg = nsegments(total_rows)
    threads = max(1, (os.cpu_count() or 1) // world)
    if writer == "oracle":
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O

        codec = O.CODEC_PFOR_INT if kind == "pfor" else O.CODEC_DENSE_INT
        write = lambda a, b, meta: O.synth_write(d, table, total_rows, BLOCK, SEGMENT, codec, a, b, meta, nthreads=threads)  # noqa: E731
    else:
        from immutable3_b200 import _lib as L
        from immutable3_b200.loader import synth_write

        os.environ.setdefault("IMM3_WRITER_THREADS", str(threads))
        codec = L.CODEC_PFOR_INT if kind == "pfor" else L.CODEC_DENSE_INT
        write = lambda a, b, meta: synth_write(d, table, total_rows, BLOCK, SEGMENT, codec, a, b, meta)  # noqa: E731
    if rank == 0:
        os.makedirs(d, exist_ok=True)
        write(0, 0, True)
    barrier()
    write(rank * nseg // world, (rank + 1) * nseg // world, False)
    barrier()
    if rank == 0:
        open(done, "w").write("ok")
    barrier()
    return d, table, time.time() - t0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(key: str):
    """dram__bytes_read+write per query from a committed ncu capture: {"bytes": ..., "source": "profiles/<file>"} or None.
    (bench.py cannot run ncu on itself; the figure is tied to the capture it names.)"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            v = json.load(open(p)).get(key)
            if isinstance(v, dict):
                return v
            if v is not None:
                return {"bytes": v, "source": "profiles/traffic.json"}
        except Exception:
            return None
    return None


def crc_columns(cols):
    import numpy as np

    return [(int(len(c)), zlib.crc32(np.ascontiguousarray(c).view(np.uint8).reshape(-1).tobytes())) for c in cols]


def dump_outputs(out_dir, names, cols, result_rows, suffix=""):
    """--dump-outputs: one query's result as out_dir/<column><suffix>.npy in float64 (a STRING(k) column as n x k byte
    codes) and its row count as result_rows<suffix>.npy.  A result above DUMP_BYTES is cut to one seeded sample of rows,
    the same in every column, whose positions go to sample_rows<suffix>.npy: two builds run with the same arguments
    can then be compared array for array."""
    import numpy as np

    arrays = {"result_rows": np.array([result_rows], np.float64)}
    per_row = sum(c.dtype.itemsize if c.dtype.kind == "S" else 1 for c in cols)  # float64 values per result row
    n = len(cols[0]) if cols else 0
    cap = (DUMP_BYTES - 4096) // (8 * (per_row + 1))  # (+1: the sample's positions; 4096: the .npy headers)
    rows = None
    if n > cap:
        rows = np.sort(np.random.default_rng(0).choice(n, size=cap, replace=False))
        arrays["sample_rows"] = rows.astype(np.float64)
    for name, c in zip(names, cols):
        if rows is not None:
            c = c[rows]
        if c.dtype.kind == "S":
            c = np.ascontiguousarray(c).view(np.uint8).reshape(len(c), c.dtype.itemsize)
        arrays[name] = c.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


# ---------------------------------------------------------------------------------------------------
# CPU side: the oracle (restatement of the reference's Scala path), one task per segment on a pool
# ---------------------------------------------------------------------------------------------------
def load_oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import build_oracle

    build_oracle.build_oracle()
    import oracle_lib as O

    return O


def run_cpu(O, d, table, workload, total_rows, nthreads, steps, warmup, seg_begin=0, seg_end=-1):
    agg = AGG_SPECS.get(workload)
    preds, proj, limit = (agg[0], None, 0) if agg else query_spec(workload, total_rows)
    times, res = [], None
    with O.Oracle(d) as orc:
        rows_scanned = orc.nrows(table, seg_begin, seg_end)
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            if agg:
                res = orc.query_agg(table, preds, agg[1], agg[2], nthreads=nthreads, seg_begin=seg_begin, seg_end=seg_end)
            else:
                res = orc.query(table, preds, proj, limit=limit, nthreads=nthreads, seg_begin=seg_begin, seg_end=seg_end)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    return rows_scanned, res, times


def config_dict(args, workload, total_rows, world, extra=None):
    c = {"workload": WORKLOADS[workload][0], "rows_total": total_rows, "rows_per_gpu": total_rows // max(1, world), "block_size": BLOCK,
         "segment_size": SEGMENT, "segments": nsegments(total_rows), "scaling": args.scaling,
         "sharding": "contiguous canonical segment slices, one per GPU (SegmentManager.scala:41 order)"}
    if extra:
        c.update(extra)
    return c


def protocol_keys(args, result_rows):
    """The measurement-protocol part of `config`: the same dict in both arms (--impl ours / reference), so that the two lines
    describe one configuration; what is specific to an arm says which arm it is about."""
    return {"l2": "GPU arm: flushed between steps (512 MiB %s pass); reference arm: the table is larger than every host cache"
                  % os.environ.get("IMM3_BENCH_FLUSH", "read"),
            "kernel_variant": "direct" if args.no_tma else "tma", "block_pruning": False,
            "timed": "GPU arm: wall: host barrier (ranks released at one instant of the host clock) -> imm3_query_begin returns (all kernels + "
                     "on-device count exchange + one sync); median of K steps of the max over ranks.  Reference arm: wall clock around one "
                     "whole-table query on all host threads; median of K steps",
            "result_rows": result_rows}


def reference_arm(args):
    """The reference's own CPU path - as far as it can exist here: the Scala engine cannot run (no JVM), so this is the
    oracle port on all host cores, same table, same query, same --steps/--warmup.  No product code is imported."""
    O = load_oracle()
    world = max(1, args.gpus)
    total = args.rows * (world if args.scaling == "weak" else 1)
    kind = WORKLOADS[args.workload][1]
    d, table, gen_s = ensure_table(kind, total, 0, 1, lambda: None, "oracle")
    cores = os.cpu_count() or 1
    rows, res, times = run_cpu(O, d, table, args.workload, total, cores, args.steps, args.warmup)
    if args.dump_outputs:
        agg = AGG_SPECS.get(args.workload)
        names = (agg[2] + [col + ("_count", "_min", "_max")[op] for op, col in agg[1]]) if agg else query_spec(args.workload, total)[1]
        dump_outputs(args.dump_outputs, names, res.columns, res.nrows)
    sec = statistics.median(times)
    v = rows / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_dict(args, args.workload, total, world, protocol_keys(args, res.nrows)),
        "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port",
                         "sample": f"whole table ({rows} rows) per step, one task per segment on {cores} threads (Engine.scala:176-180); "
                                   "CPU restatement of the reference path - the Scala engine itself cannot run here (no JVM)"},
        "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "result_rows": res.nrows, "table_gen_s": gen_s,
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=list(WORKLOADS))
    ap.add_argument("--rows", type=int, default=None, help="rows of the table (strong scaling: total; weak: per GPU); default 1e9 for the "
                                                            "test_1b workloads, 1e8 for the test_100m ones")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="C5: the selectivity sweep on test_1b (id windows 0.01 % .. 100 %, age < t, state + age), "
                    "LIMIT 10 vs none, instead of the headline run; one JSON line with a `sweep` table")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-tma", action="store_true", help="direct-load variant of the dense kernels (A/B)")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the rows the last timed step computed to DIR/<column>.npy (float64, "
                    "a seeded sample of them beyond 64 MB) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.sweep:
        ap.error("--dump-outputs writes the headline query's result; --sweep has none")
    if args.rows is None:
        args.rows = 1_000_000_000 if WORKLOADS[args.workload][1] == "pfor" else 100_000_000
    if args.warmup < 3 and args.impl == "ours" and not os.environ.get("IMM3_BENCH_ALLOW_SHORT"):
        args.warmup = max(args.warmup, 3)  # timing rule: W >= 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return reference_arm(args) if rank == 0 else 0

    # ------------------------------------------------------------------ GPU arm
    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the scan path has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))  # bootstrap + result reductions only
        barrier = lambda: (torch.cuda.synchronize(), dist.barrier(), torch.cuda.synchronize())  # noqa: E731
    else:
        barrier = lambda: torch.cuda.synchronize()  # noqa: E731

    from immutable3_b200 import OPEN_KEEP_HOST, OPEN_NO_TMA, Engine, SegmentManager, flatten_select

    flush_buf = torch.zeros(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    flush_sink = torch.zeros((), dtype=torch.int64, device="cuda")
    flush_mode = os.environ.get("IMM3_BENCH_FLUSH", "read")

    def flush_l2(i):
        # Evict the table from the 126 MB L2 between steps.  A READ pass over 512 MiB leaves clean lines behind; a write
        # pass (fill_) would leave ~126 MB of dirty lines whose write-back is then charged to the next query.
        if flush_mode == "write":
            flush_buf.fill_(i & 0xFF)
        elif flush_mode == "read":
            flush_sink.copy_(flush_buf.view(torch.int64).sum())
        torch.cuda.synchronize()

    def aligned_start():
        """Host barrier, then every rank spins to the same instant of the host's monotonic clock (all ranks are processes on
        one host): the ranks leave a collective barrier tens of microseconds apart, which a 0.1 ms query would be charged
        as waiting time in the count exchange."""
        barrier()
        if world > 1:
            t = torch.tensor([time.monotonic_ns() + 300_000], dtype=torch.int64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            target = int(t.item())
        else:
            target = time.monotonic_ns() + 20_000
        while time.monotonic_ns() < target:
            pass

    def allmax(values):
        if world == 1:
            return list(values)
        t = torch.tensor(list(values), dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def allsum(v):
        if world == 1:
            return int(v)
        t = torch.tensor([int(v)], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        return int(t.item())

    opened = {}  # (kind, rows) -> (sm, eng, dir, table, tinfo, open_s, gen_s)

    def open_table(kind, rows_total):
        key = (kind, rows_total)
        if key not in opened:
            d, table, gen_s = ensure_table(kind, rows_total, rank, world, barrier, "product")
            flags = OPEN_KEEP_HOST | (OPEN_NO_TMA if args.no_tma else 0)  # (KEEP_HOST: a pinned mirror is built on the first reupload only)
            barrier()
            t0 = time.perf_counter()
            sm = SegmentManager(d, device=local_rank, rank=rank, world=world, flags=flags)
            open_s = time.perf_counter() - t0
            if world > 1:
                sm.comm_connect()  # the GPUs exchange the per-rank counts themselves from here on (imm3_comm_*)
            opened[key] = (sm, Engine(sm), d, table, sm.getTable(table), open_s, gen_s)
        return opened[key]

    def measure(workload, rows_total, steps, warmup, sample_clocks=False, prune=False, outputs=None):
        """K timed steps of one query.  Per step: L2 flush + barrier (untimed), then the wall time of imm3_query_begin -
        launch of every kernel of the query, the on-device count exchange, one synchronisation, counts on the host.
        `outputs` (a dict) receives the result of the last step, fetched after its clock stopped."""
        sm, eng, d, table, tinfo, open_s, gen_s = open_table(WORKLOADS[workload][1], rows_total)
        query = build_query(workload, table, rows_total)
        is_agg = workload in AGG_SPECS
        prep = None if is_agg else eng.prepare(query)
        run = (lambda: eng.execute(query)) if is_agg else (lambda: eng.begin_prepared(prep))
        # Block pruning (per-block min/max, SURVEY.md 8f-4) changes the bytes a range query on the encoded column has to read:
        # the headline is the plain scan (every block decided from its encoded bytes); the pruned figure is a secondary record.
        if os.environ.get("IMM3_BENCH_KEEP_PRUNE_ENV"):
            pass  # (profiling scripts choose the mode themselves)
        elif prune:
            os.environ.pop("IMM3_NO_PRUNE", None)
        else:
            os.environ["IMM3_NO_PRUNE"] = "1"
        wall, dev, launches, alg, local_rows, take, gcount = [], [], 0, 0, 0, 0, 0
        phases = []
        for i in range(warmup):
            flush_l2(i)
            aligned_start()
            run().close()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        for i in range(steps):
            flush_l2(i)
            aligned_start()
            t0 = time.perf_counter()
            r = run()
            t1 = time.perf_counter()
            wall.append((t1 - t0) * 1e3)
            dev.append(r.device_ms)
            phases.append(r.host_us())
            launches += r.kernel_launches
            alg, local_rows, take, gcount = r.algorithmic_bytes, r.local_count, r.take, r.global_count
            if outputs is not None and i == steps - 1:
                if not is_agg:
                    r.fetch(r.take)  # (an aggregate's rows are on the host already)
                outputs.update(names=[r.col_name(c) for c in range(r.ncols)], cols=r.columns(), result_rows=gcount)
            r.close()
        clocks = sampler.stop() if sampler else None
        barrier()
        wall_max, dev_max = allmax(wall), allmax(dev)
        ms = statistics.median(wall_max)
        rec = {"workload": WORKLOADS[workload][0], "rows_total": rows_total, "value": rows_total / (ms * 1e-3), "unit": "rows/s",
               "ms_per_step": ms, "wall_ms": {"median": ms, "mean": statistics.mean(wall_max), "min": min(wall_max), "max": max(wall_max)},
               "device_ms": {"median": statistics.median(dev_max), "mean": statistics.mean(dev_max), "min": min(dev_max)},
               "host_overhead_us": (ms - statistics.median(dev_max)) * 1e3, "result_rows": gcount,
               "host_phase_us_rank0": dict(zip(("plan", "buffers+device_plan", "launches", "wait_gpu", "epilogue"),
                                               [statistics.median(p[i] for p in phases) for i in range(5)])),
               "gpu_launches": allsum(launches), "steps": steps, "block_pruning": bool(prune)}
        # roofline of the query's kernels (rank 0's slice: its algorithmic bytes / its CUDA-event time)
        peak, peak_src = measured_peak()
        my_ms = statistics.mean(dev)
        rec["roofline"] = {"bound": "hbm", "achieved": alg / (my_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": alg / (my_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg, "launch_ms_mean": my_ms,
                           "launch_ms_min": min(dev), "peak_source": peak_src, "slice": f"rank 0 of {world}"}
        return rec, clocks, (sm, eng, d, table, tinfo, query, prep, local_rows, take)

    def stage_times(eng, prep, n=5):
        """Per-kernel CUDA-event times: the emit kernel normally is a programmatic dependent launch of the filter kernel (no
        event may sit between them), so a few extra UNTIMED queries run with IMM3_NO_PDL=1."""
        os.environ["IMM3_NO_PDL"] = "1"
        a, b = [], []
        try:
            for i in range(n + 1):
                flush_l2(i)
                barrier()
                with eng.begin_prepared(prep) as r:
                    if i:
                        a.append(r.stage_ms(0))
                        b.append(r.stage_ms(1))
        finally:
            os.environ.pop("IMM3_NO_PDL", None)
        return statistics.mean(a), statistics.mean(b)

    def verify(O, workload, rows_total, ctx, nthreads, oracle_result=None):
        """Content parity at full size: this rank's fetched rows vs the oracle over this rank's slice (CRC-32 per column)."""
        sm, eng, d, table, tinfo, query, prep, _, _ = ctx
        if workload in AGG_SPECS:
            # per-rank partial aggregates vs the oracle over this rank's slice (groups, order and values)
            with eng.execute(query) as r:
                got = crc_columns(r.columns())
            _, ores, _ = run_cpu(O, d, table, workload, rows_total, nthreads, 1, 0, tinfo.seg_begin, tinfo.seg_end)
            return got == crc_columns(ores.columns)
        with eng.begin_prepared(prep) as r:
            r.fetch(r.take)
            got = crc_columns(r.columns())
            take, offset = r.take, r.global_offset
            counts = r.rank_counts
        if oracle_result is None:
            _, oracle_result, _ = run_cpu(O, d, table, workload, rows_total, nthreads, 1, 0, tinfo.seg_begin, tinfo.seg_end)
        want = crc_columns([c[:take] for c in oracle_result.columns])
        limit = int(query.project.limit)
        ok = got == want and (limit > 0 or take == oracle_result.nrows) and offset == sum(counts[:rank])
        return bool(ok)

    # ---- C5: the selectivity sweep (its own JSON line; the headline protocol per point, fewer steps) ----
    if args.sweep:
        cores = os.cpu_count() or 1
        total = args.rows * (world if args.scaling == "weak" else 1)
        table = []
        peak, peak_src = measured_peak()
        for wl in SWEEP:
            for lim in ("", "_limit10"):
                name = wl + lim
                try:
                    rec, _, sctx = measure(name, total, max(5, args.steps // 2), 3, prune=True)  # (the library's defaults: pruning on)
                    row = {"point": name, "query": WORKLOADS[name][0], "result_rows": rec["result_rows"], "selectivity": rec["result_rows"] / total if not lim else None,
                           "wall_ms": rec["ms_per_step"], "device_ms": rec["device_ms"]["median"], "rows_per_s": rec["value"],
                           "gpu_launches_per_query": rec["gpu_launches"] / max(1, rec["steps"]) / world,
                           # (A = the full scan's bytes: no roofline figure for LIMIT points - a prefix of the table is read - nor for pruned
                           #  id windows - 8 B of statistics per block are read instead of the column: see "unpruned")
                           "roofline_frac_rank0": None if (lim or name.startswith("c5w_")) else rec["roofline"]["frac"],
                           "algorithmic_bytes_rank0": rec["roofline"]["algorithmic_bytes_per_launch"]}
                    if not lim and name.startswith("c5w_"):  # id windows: also the plain scan (every block decided from its encoded bytes)
                        rec2, _, _ = measure(name, total, max(5, args.steps // 2), 3, prune=False)
                        row["unpruned"] = {"wall_ms": rec2["ms_per_step"], "device_ms": rec2["device_ms"]["median"], "rows_per_s": rec2["value"],
                                           "roofline_frac_rank0": rec2["roofline"]["frac"]}
                    if not args.no_verify and rec["result_rows"] <= 110_000_000:
                        ok = verify(load_oracle(), name, total, sctx, max(1, cores // world))
                        if world > 1:
                            everyone = [None] * world
                            dist.all_gather_object(everyone, ok)
                            ok = all(everyone)
                        row["result_equal"] = ok
                    table.append(row)
                except Exception as e:
                    table.append({"point": name, "error": repr(e)})
        if rank == 0:
            pts = [r for r in table if "rows_per_s" in r]
            print(json.dumps({"metric": METRIC, "value": statistics.median([r["rows_per_s"] for r in pts]) if pts else None, "unit": "rows/s", "n_gpus": world,
                              "steps": max(5, args.steps // 2), "warmup": 3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                              "dtype": "u8", "data": "synthetic",
                              "config": {"workload": "C5 selectivity sweep on test_1b (id:PFOR_INT, state:DENSE_STRING:2, age:DENSE_TINYINT), LIMIT 10 vs none",
                                         "rows_total": total, "segments": nsegments(total), "sharding": "contiguous canonical segment slices, one per GPU",
                                         "l2": "flushed between steps", "value_is": "median rows/s over the sweep points (wall: barrier -> query + count exchange done)",
                                         "peak_gbs": peak, "peak_source": peak_src},
                              "sweep": table}))
        for v in opened.values():
            v[0].close()
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- headline: value = wall (barrier -> query + exchange done), K steps ----
    total = args.rows * (world if args.scaling == "weak" else 1)
    outputs = {} if args.dump_outputs else None
    head, clocks, ctx = measure(args.workload, total, args.steps, args.warmup, sample_clocks=True, outputs=outputs)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs["names"], outputs["cols"], outputs["result_rows"], f"_rank{rank}" if world > 1 else "")
    sm, eng, d, table, tinfo, query, prep, local_rows, take = ctx
    open_s, gen_s = opened[(WORKLOADS[args.workload][1], total)][5:7]
    agg_head = args.workload in AGG_SPECS
    st0, st1 = (None, None) if (agg_head or os.environ.get("IMM3_BENCH_NO_STAGES")) else stage_times(eng, prep)
    kind = WORKLOADS[args.workload][1]
    on_pfor_filter = kind == "pfor" and any(l.col == "id" for l in flatten_select(query.select))
    kname = ("filter_kernel -> agg_kernel -> agg_compact_kernel" if agg_head else
             ("blocks_filter_lane_kernel (sorted-int codec, one lane per block, per-warp TMA rings) -> blocks_group_emit_kernel (emit from per-group sums, no offset scan)"
              if list(query.project.cols) == ["id"] else
              "blocks_filter_lane_kernel (sorted-int codec, one lane per block) [-> offset_scan_kernel] -> blocks_emit_kernel") if on_pfor_filter else
             "filter_kernel (row space) -> blocks_emit_kernel" if kind == "pfor" else "filter_kernel -> emit_stream_kernel | emit_kernel")
    roofline = head.pop("roofline")
    tr = recorded_traffic(f"{args.workload}_{total}") if world == 1 else None
    roofline.update({"kernel": kname + " (one query = one launch of each; timed together with CUDA events)",
                     "stage_ms_mean": {"filter (+ offset scan where it is a kernel of its own)": st0, "emit (blocks_group_emit_kernel on the headline path)": st1,
                                       "note": "from an extra IMM3_NO_PDL=1 pass (kernels serialised, an event between them)"},
                     "traffic": tr["bytes"] if tr else None, "traffic_source": ("ncu capture " + tr["source"]) if tr else None})

    # ---- e2e through the C ABI ----
    used_cols = sorted({l.col for l in flatten_select(query.select)} | (set() if agg_head else set(query.project.cols)))
    used_bytes = allsum(sum(c.encoded_bytes for c in tinfo.columns if c.name in used_cols))

    def e2e_pass(reupload: bool):
        """K steps back to back, timed as a whole.  Every step stages its inputs (H2D), runs the query (count exchange on
        the device) and reads this rank's share of the result rows back (D2H); the read-back of step i is asynchronous and
        overlaps the staging of step i+1 (full-duplex PCIe); every result is waited for before the clock stops."""
        w_e2e = max(2, args.warmup // 2)
        d2h, t0, prev = 0, 0.0, None
        for i in range(w_e2e + args.steps):
            if i == w_e2e:
                if prev is not None:
                    prev.wait().close()
                    prev = None
                sm.sync()
                barrier()
                t0 = time.perf_counter()
            if reupload:
                sm.reupload(table, used_cols)          # H2D of this step's inputs from pinned host memory (async)
            r = eng.begin_prepared(prep)               # kernels + count exchange; returns when the counts are on the host
            r.fetch_async(r.take)                      # result rows -> pinned host buffers, on the copy stream
            if prev is not None:
                prev.wait()
                prev.close()
            prev = r
        prev.wait()
        d2h = sum(prev.col_width(c) for c in range(prev.ncols)) * prev.nrows
        assert prev.nrows == prev.take
        prev.close()
        sm.sync()
        barrier()
        dt = time.perf_counter() - t0
        return allmax([dt])[0] / args.steps, allsum(d2h)

    e2e = e2e_res = None
    if not args.no_e2e and not agg_head:
        sec_res, d2h_b = e2e_pass(False)
        sec_cold, _ = e2e_pass(True)
        e2e = {"value": total / sec_cold, "unit": "rows/s", "h2d_bytes_per_step": used_bytes, "d2h_bytes_per_step": d2h_b,
               "ms_per_step": sec_cold * 1e3,
               "what": "per step: re-stage the query's columns host(pinned)->HBM, kernels + on-device count exchange, this rank's result rows -> host "
                       "(read-back of step i overlaps the staging of step i+1; K steps timed as a whole, max over ranks)"}
        e2e_res = {"value": total / sec_res, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h_b, "ms_per_step": sec_res * 1e3,
                   "what": "table resident in HBM (SegmentManager loads once): kernels + count exchange, result rows -> host"}

    # ---- CPU baseline beside it (rank 0, N=1 only) + content parity on every rank ----
    cpu, result_equal = None, None
    cores = os.cpu_count() or 1
    if not args.no_verify or (world == 1 and not args.no_cpu_baseline):
        O = load_oracle()
        oracle_res = None
        if world == 1 and not args.no_cpu_baseline:
            rows, oracle_res, times = run_cpu(O, d, table, args.workload, total, cores, args.cpu_steps, 1)
            cpu = {"value": rows / statistics.mean(times), "unit": "rows/s", "cores": cores, "kind": "port",
                   "sample": f"whole table ({rows} rows), {args.cpu_steps} passes after 1 warm-up, one task per segment on {cores} threads"}
        if not args.no_verify:
            mine = verify(O, args.workload, total, ctx, max(1, cores // world), oracle_res)
            if world > 1:
                everyone = [None] * world
                dist.all_gather_object(everyone, mine)
                result_equal = everyone
            else:
                result_equal = [mine]
            if cpu is not None:
                cpu["result_equal"] = mine

    # ---- secondary records (same protocol, fewer steps) ----
    secondary = {}
    if not args.no_secondary and args.workload == "c4":
        for name, wl, rows in SECONDARY:
            rows_total = (rows if rows is not None else args.rows) * (world if args.scaling == "weak" else 1)
            try:
                rec, _, sctx = measure(wl, rows_total, max(5, args.steps // 2), 3, prune=True)  # (secondary records: the library's defaults)
                if not args.no_verify and rec["result_rows"] <= 50_000_000:
                    ok = verify(load_oracle(), wl, rows_total, sctx, max(1, cores // world))
                    if world > 1:
                        everyone = [None] * world
                        dist.all_gather_object(everyone, ok)
                        ok = everyone
                    rec["result_equal"] = ok
                secondary[name] = rec
            except Exception as e:  # a secondary record must never cost the headline
                secondary[name] = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": config_dict(args, args.workload, total, world, protocol_keys(args, head["result_rows"])),
            "clocks": clocks, "timing": {k: head[k] for k in ("wall_ms", "device_ms", "host_overhead_us", "host_phase_us_rank0")},
            "e2e": e2e, "e2e_resident": e2e_res, "gpu_launches": head["gpu_launches"], "roofline": roofline, "cpu_baseline": cpu,
            "result_equal": result_equal, "workloads": secondary, "open_s": open_s,
            "upload_gbs": tinfo.resident_bytes / open_s / 1e9, "resident_bytes_rank0": tinfo.resident_bytes, "table_gen_s": gen_s,
        }
        print(json.dumps(line))
    for v in opened.values():
        v[0].close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
