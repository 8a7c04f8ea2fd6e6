"""SUM / AVG aggregates (imm3_query_agg_ext: the SUM instantiations of agg_kernel / agg_blocks_kernel) against COUNT / MIN /
MAX queries of the same plan width on the same tables.

  S1 / C1  test_100m (dense): sum(age), avg(age) where age > 18 group by state  vs  count(age), min(age), max(age) - both
           run a plan of three aggregates (S1: the SUM, the AVG's SUM and the hidden COUNT)
  S2       test_1b (id:PFOR_INT, agg_blocks_kernel) and its dense-id twin (agg_kernel): sum(id), avg(age) group by state
  G*       the same through IMM3_AGG_GLOBAL on a world == 1 handle
bench.py's tables and the protocol of tools/agg_encoded_bench.py: >= 3 warm-up and >= 20 timed steps per query, the L2
evicted by a 512 MiB read pass before each, median and min of the CUDA-event time of the query's kernels (Result.device_ms)
and of the wall time of Engine.execute.  Checks: S1's sums and averages against numpy over the oracle's selected rows
(exact: the sums stay below 2^53), every group set and count against the oracle's query_agg, S2 between the twins, every
G* against its local form.  The GPU's name and power limit are read in the same run.

usage: python tools/agg_sum_bench.py [--rows-small N] [--rows N] [--steps K] [--warmup W] [--out profiles/<name>.json]"""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows-small", type=int, default=100_000_000)
    ap.add_argument("--rows", type=int, default=1_000_000_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_agg_sum.json"))
    args = ap.parse_args()
    args.steps, args.warmup = max(20, args.steps), max(3, args.warmup)

    import numpy as np
    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the aggregation kernels have no CPU fallback"}))
        return 2
    import oracle_lib as O
    from immutable3_b200 import GT, Avg, Count, Engine, Max, Min, NoSelect, ProjectAgg, Query, SegmentManager, Select, Sum

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    flush_buf = torch.zeros(512 << 20, dtype=torch.uint8, device="cuda")
    flush_sink = torch.zeros((), dtype=torch.int64, device="cuda")

    def flush_l2():
        flush_sink.copy_(flush_buf.view(torch.int64).sum())
        torch.cuda.synchronize()

    def timed(eng, q, glob, sum_avg):
        run = (lambda: eng.execute_agg_global(q, sum_avg=sum_avg)) if glob else (lambda: eng.execute(q, sum_avg=sum_avg))
        wall, dev = [], []
        for i in range(args.warmup + args.steps):
            flush_l2()
            t0 = time.perf_counter()
            r = run()
            t1 = time.perf_counter()
            if i >= args.warmup:
                wall.append((t1 - t0) * 1e3)
                dev.append(r.device_ms)
            if i == args.warmup + args.steps - 1:
                cols, route, alg = [np.asarray(c) for c in r.columns()], r.route, r.algorithmic_bytes
            r.close()
        rec = {"groups": int(len(cols[0])) if cols else 0, "route": route, "algorithmic_bytes": alg,
               "device_ms": {"median": statistics.median(dev), "min": min(dev)}, "wall_ms": {"median": statistics.median(wall), "min": min(wall)}}
        return rec, cols

    cores = os.cpu_count() or 1
    sel = Select("age", GT(18))
    out = {"gpu": gpu, "steps": args.steps, "warmup": args.warmup,
           "protocol": "per step: 512 MiB read pass (L2 eviction), then Engine.execute; device = CUDA events around the query's kernels",
           "queries": {"S1": "select sum(age), avg(age) from test_100m where age > 18 group by state",
                       "C1": "select count(age), min(age), max(age) from test_100m where age > 18 group by state",
                       "S2": "select sum(id), avg(age) from test_1b group by state (pfor: encoded id, dense: the dense-id twin)"},
           "checks": {}, "records": {}}

    # S1 / C1 at --rows-small on the dense table
    d, table, _ = bench.ensure_table("dense", args.rows_small, 0, 1, lambda: None, "product")
    s1 = Query(table, sel, ProjectAgg([Sum("age"), Avg("age")], ["state"]))
    c1 = Query(table, sel, ProjectAgg([Count("age"), Min("age"), Max("age")], ["state"]))
    with SegmentManager(d) as sm, O.Oracle(d) as orc:
        eng = Engine(sm)
        for name, q, sa in (("S1", s1, True), ("C1", c1, False)):
            for glob in (False, True):
                rec, cols = timed(eng, q, glob, sa)
                out["records"][("G" if glob else "") + name + f"_{args.rows_small // 1_000_000}m"] = rec
                print(name, glob, json.dumps(rec), flush=True)
                if name == "S1":
                    if not glob:
                        s1_cols = cols
                    else:
                        out["checks"]["GS1_equals_S1"] = all(a.tobytes() == b.tobytes() for a, b in zip(cols, s1_cols))
                else:
                    exp = orc.query_agg(table, [("age", O.OP_GT, 18)], [(O.AGG_COUNT, "age"), (O.AGG_MIN, "age"), (O.AGG_MAX, "age")], ["state"], nthreads=cores)
                    out["checks"][("G" if glob else "") + "C1_oracle_equal"] = all(np.array_equal(a, b) for a, b in zip(cols, exp.columns))
                    if not glob:
                        c1_cols = cols
        rows = orc.query(table, [("age", O.OP_GT, 18)], ["state", "age"], limit=0, nthreads=cores)
        st, age = np.asarray(rows.columns[0]), np.asarray(rows.columns[1]).astype(np.int64)
        keys, first, inv = np.unique(st, return_index=True, return_inverse=True)
        order = np.argsort(first)
        rank = np.empty_like(order)
        rank[order] = np.arange(len(order))
        g = rank[inv.reshape(-1)]
        cnt = np.bincount(g)
        sums = np.bincount(g, weights=age.astype(np.float64)).astype(np.int64)  # exact: every sum < 2^53
        out["checks"]["S1_numpy_equal"] = (list(s1_cols[0]) == list(keys[order]) and s1_cols[1].tolist() == sums.tolist()
                                           and s1_cols[2].tobytes() == (sums.astype(np.float64) / cnt.astype(np.float64)).tobytes())
        out["checks"]["S1_groups_equal_C1"] = list(s1_cols[0]) == list(c1_cols[0])
    # S2 at --rows on the encoded table and its dense twin
    s2_cols = {}
    for kind in ("pfor", "dense"):
        d, table, _ = bench.ensure_table(kind, args.rows, 0, 1, lambda: None, "product")
        q = Query(table, NoSelect, ProjectAgg([Sum("id"), Avg("age"), Count("id")], ["state"]))
        with SegmentManager(d) as sm, O.Oracle(d) as orc:
            eng = Engine(sm)
            q2 = Query(table, NoSelect, ProjectAgg([Sum("id"), Avg("age")], ["state"]))
            for glob in (False, True):
                rec, cols = timed(eng, q2, glob, True)
                out["records"][("G" if glob else "") + f"S2_{kind}_{args.rows // 1_000_000}m"] = rec
                print(kind, glob, json.dumps(rec), flush=True)
                if glob:
                    out["checks"][f"GS2_{kind}_equals_S2"] = all(a.tobytes() == b.tobytes() for a, b in zip(cols, s2_cols[kind]))
                else:
                    s2_cols[kind] = cols
            with eng.execute(q, sum_avg=True) as r:
                cnt = np.asarray(r.column(3))
            exp = orc.query_agg(table, [], [(O.AGG_COUNT, "id")], ["state"], nthreads=cores)
            out["checks"][f"S2_{kind}_groups_and_counts_oracle_equal"] = (list(s2_cols[kind][0]) == list(exp.columns[0])
                                                                          and cnt.tolist() == np.asarray(exp.columns[1]).tolist())
    out["checks"]["S2_twins_equal"] = all(a.tobytes() == b.tobytes() for a, b in zip(s2_cols["pfor"], s2_cols["dense"]))
    out["s1_over_c1_device_median"] = out["records"][f"S1_{args.rows_small // 1_000_000}m"]["device_ms"]["median"] / \
        out["records"][f"C1_{args.rows_small // 1_000_000}m"]["device_ms"]["median"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "checks", "s1_over_c1_device_median")}))
    return 0 if all(out["checks"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
