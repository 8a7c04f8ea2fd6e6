"""Aggregation over a sorted-int-codec column (agg_blocks_kernel) against the same queries on the dense-id twin (agg_kernel).

test_1b (id:PFOR_INT) and its dense twin (id:DENSE_INT, same rows) at the same size, bench.py's tables and protocol: >= 3 warm-up
and >= 20 timed steps per query, the L2 evicted by a 512 MiB read pass before each, median and min of the CUDA-event time of the
query's kernels (Result.device_ms) and of the wall time of Engine.execute.  Every query's groups are checked against the oracle
(oracle_lib.Oracle.query_agg) on the same files and between the twins; a separate torch.profiler pass per query gives each
kernel's time.  The GPU's name and power limit are read in the same run.

usage: python tools/agg_encoded_bench.py [--rows N] [--steps K] [--warmup W] [--out profiles/<name>.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402

# name: (what, predicates as (col, op, value) with op 1 = GT, 4 = MATCH, aggregates as (op, col) with op 0 / 1 / 2 = count / min / max, group by)
QUERIES = {
    "Q1": ("select count(id), min(id), max(id) from T where age > 18 group by state (81 % of rows: every block decoded)",
           [("age", 1, 18)], [(0, "id"), (1, "id"), (2, "id")], ["state"]),
    "Q2": ("select min(id), max(id) from T where state = 'CA' group by age (~2 %, scattered)",
           [("state", 4, ["CA"])], [(1, "id"), (2, "id")], ["age"]),
    "Q3": ("select min(id), max(id), count(age) from T (no predicate)",
           [], [(1, "id"), (2, "id"), (0, "age")], []),
}


def build_query(table, spec):
    from immutable3_b200 import GT, And, Count, Match, Max, Min, NoSelect, ProjectAgg, Query, Select

    _, preds, aggs, group_by = spec
    sel = NoSelect
    for i, (c, op, v) in enumerate(preds):
        leaf = Select(c, GT(v)) if op == 1 else Select(c, Match(v))
        sel = leaf if i == 0 else And(sel, leaf)
    return Query(table, sel, ProjectAgg([{0: Count, 1: Min, 2: Max}[op](col) for op, col in aggs], group_by))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_agg_encoded.json"))
    args = ap.parse_args()
    args.steps, args.warmup = max(20, args.steps), max(3, args.warmup)

    import numpy as np
    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the aggregation kernels have no CPU fallback"}))
        return 2
    import oracle_lib as O
    from immutable3_b200 import Engine, SegmentManager

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    flush_buf = torch.zeros(512 << 20, dtype=torch.uint8, device="cuda")
    flush_sink = torch.zeros((), dtype=torch.int64, device="cuda")

    def flush_l2():
        flush_sink.copy_(flush_buf.view(torch.int64).sum())  # a READ pass: no dirty lines left for the query to write back
        torch.cuda.synchronize()

    cores = os.cpu_count() or 1
    out = {"gpu": gpu, "rows": args.rows, "steps": args.steps, "warmup": args.warmup,
           "protocol": "per step: 512 MiB read pass (L2 eviction), then Engine.execute; device = CUDA events around the query's kernels",
           "tables": {}, "queries": {k: v[0] for k, v in QUERIES.items()}}
    results = {}
    for kind in ("pfor", "dense"):
        d, table, gen_s = bench.ensure_table(kind, args.rows, 0, 1, lambda: None, "product")
        sm = SegmentManager(d)
        eng = Engine(sm)
        rec = {"table": table, "id_codec": "PFOR_INT" if kind == "pfor" else "DENSE_INT", "table_gen_s": gen_s}
        with O.Oracle(d) as orc:
            for name, spec in QUERIES.items():
                q = build_query(table, spec)
                wall, dev = [], []
                for i in range(args.warmup + args.steps):
                    flush_l2()
                    t0 = time.perf_counter()
                    r = eng.execute(q)
                    t1 = time.perf_counter()
                    if i >= args.warmup:
                        wall.append((t1 - t0) * 1e3)
                        dev.append(r.device_ms)
                    if i == args.warmup + args.steps - 1:
                        cols = [np.asarray(c) for c in r.columns()]
                        alg = r.algorithmic_bytes
                    r.close()
                # per-kernel times (a run of its own: the profiler slows the host)
                from torch.profiler import ProfilerActivity, profile

                flush_l2()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(5):
                        flush_l2()
                        eng.execute(q).close()
                kern = {}
                for e in prof.key_averages():
                    if "kernel" in e.key and ("agg" in e.key or "filter" in e.key):
                        t = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
                        kern[e.key.split("(")[0].replace("void ", "").replace("imm3::", "")] = round(t / 1e3, 4)  # mean ms per launch
                exp = orc.query_agg(table, spec[1], spec[2], spec[3], nthreads=cores)
                oracle_ok = len(cols) == len(exp.columns) and all(np.array_equal(a, b) for a, b in zip(cols, exp.columns))
                results[(kind, name)] = cols
                rec[name] = {"groups": int(len(cols[0])) if cols else 0, "device_ms": {"median": statistics.median(dev), "min": min(dev)},
                             "wall_ms": {"median": statistics.median(wall), "min": min(wall)}, "algorithmic_bytes": alg,
                             "kernel_ms_mean": kern, "oracle_equal": bool(oracle_ok)}
                print(kind, name, json.dumps(rec[name]), flush=True)
        sm.close()
        out["tables"][kind] = rec
    out["twin_equal"] = {name: all(np.array_equal(a, b) for a, b in zip(results[("pfor", name)], results[("dense", name)]))
                         and len(results[("pfor", name)]) == len(results[("dense", name)]) for name in QUERIES}
    out["pfor_over_dense_device_median"] = {name: out["tables"]["pfor"][name]["device_ms"]["median"] / out["tables"]["dense"][name]["device_ms"]["median"]
                                            for name in QUERIES}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "twin_equal", "pfor_over_dense_device_median")}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
