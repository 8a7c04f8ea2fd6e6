"""Aggregates under a window on the sorted-int-codec id (imm3_query_agg_ext with IMM3_AGG_ENCODED_FILTER: the block filter
front - blocks_prune, the lane / mini-block filter kernel - feeding agg_blocks_kernel<.., BS = true>) against the same
queries on the dense-id twin, which stream the id column through the row-space filter kernel.

  W<p>_pfor / W<p>_pfor_noprune / W<p>_dense   select count(id), min(age), max(age) from test_1b where id > L and id < H
                                               group by state, the window holding about p % of the rows (p = 1, 10, 50, 100);
                                               pruned (default), IMM3_NO_PRUNE=1, and on the dense twin
  M10_*                                        the 10 % window and age > 18 (mini-block kernel, unpruned, on the encoded table)
  S10_*                                        sum(age), avg(age) with the 10 % window
bench.py's tables and the protocol of tools/agg_encoded_bench.py: >= 3 warm-up and >= 20 timed steps per query, the L2
evicted by a 512 MiB read pass before each, median and min of the CUDA-event time of the query's kernels (Result.device_ms)
and of the wall time of Engine.execute.  Checks: W10_pfor against the oracle's query_agg, and every query's columns equal
across the encoded table pruned / unpruned and the dense twin.  The GPU's name and power limit are read in the same run.

usage: python tools/agg_encoded_filter_bench.py [--rows N] [--steps K] [--warmup W] [--out profiles/<name>.json]"""
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
    ap.add_argument("--rows", type=int, default=1_000_000_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-oracle", action="store_true", help="skip the oracle check (the twins are still compared)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_agg_encoded_filter.json"))
    args = ap.parse_args()
    args.steps, args.warmup = max(20, args.steps), max(3, args.warmup)

    import numpy as np
    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the aggregation kernels have no CPU fallback"}))
        return 2
    import oracle_lib as O
    from helpers import conj, oracle_preds
    from immutable3_b200 import GT, LT, Avg, Count, Engine, Max, Min, NoSelect, ProjectAgg, Query, SegmentManager, Select, Sum

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    flush_buf = torch.zeros(512 << 20, dtype=torch.uint8, device="cuda")
    flush_sink = torch.zeros((), dtype=torch.int64, device="cuda")

    def flush_l2():
        flush_sink.copy_(flush_buf.view(torch.int64).sum())
        torch.cuda.synchronize()

    def timed(eng, q, sum_avg, noprune):
        if noprune:
            os.environ["IMM3_NO_PRUNE"] = "1"
        wall, dev = [], []
        try:
            for i in range(args.warmup + args.steps):
                flush_l2()
                t0 = time.perf_counter()
                r = eng.execute(q, sum_avg=sum_avg, encoded_filter=True)
                t1 = time.perf_counter()
                if i >= args.warmup:
                    wall.append((t1 - t0) * 1e3)
                    dev.append(r.device_ms)
                if i == args.warmup + args.steps - 1:
                    cols, route, alg = [np.asarray(c) for c in r.columns()], r.route, r.algorithmic_bytes
                r.close()
        finally:
            os.environ.pop("IMM3_NO_PRUNE", None)
        rec = {"groups": int(len(cols[0])) if cols else 0, "route": route, "algorithmic_bytes": alg,
               "device_ms": {"median": statistics.median(dev), "min": min(dev)}, "wall_ms": {"median": statistics.median(wall), "min": min(wall)}}
        return rec, cols

    out = {"gpu": gpu, "rows": args.rows, "steps": args.steps, "warmup": args.warmup,
           "protocol": "per step: 512 MiB read pass (L2 eviction), then Engine.execute(..., encoded_filter=True); device = CUDA events around "
                       "the query's kernels; wall = Engine.execute",
           "queries": {"W": "select count(id), min(age), max(age) from test_1b where id > L and id < H group by state",
                       "M": "the same with the 10 % window and age > 18",
                       "S": "select sum(age), avg(age) from test_1b where id > L and id < H group by state (10 % window)"},
           "windows": {}, "checks": {}, "records": {}}
    # the window bounds: the id range of the encoded table (the twins hold the same ids), split around its middle
    d_p, t_p, _ = bench.ensure_table("pfor", args.rows, 0, 1, lambda: None, "product")
    d_d, t_d, _ = bench.ensure_table("dense", args.rows, 0, 1, lambda: None, "product")
    with SegmentManager(d_p) as sm:
        with Engine(sm).execute(Query(t_p, NoSelect, ProjectAgg([Min("id"), Max("id")], []))) as r:
            lo, hi = int(r.column(0)[0]), int(r.column(1)[0])
    wins = {}
    for pct in (1, 10, 50, 100):
        if pct == 100:
            wins[pct] = (lo - 1, hi + 1)
        else:
            mid, half = (lo + hi) // 2, (hi - lo) * pct // 200
            wins[pct] = (mid - half, mid + half)
        out["windows"][str(pct)] = list(wins[pct])
    win = lambda pct: conj(Select("id", GT(wins[pct][0])), Select("id", LT(wins[pct][1])))  # noqa: E731
    cma = [Count("id"), Min("age"), Max("age")]
    plan = [("W%d" % p, win(p), cma, False) for p in (1, 10, 50, 100)]
    plan += [("M10", conj(win(10), Select("age", GT(18))), cma, False), ("S10", win(10), [Sum("age"), Avg("age")], True)]
    cols = {}
    for kind, d, table in (("pfor", d_p, t_p), ("dense", d_d, t_d)):
        with SegmentManager(d) as sm:
            eng = Engine(sm)
            for name, sel, aggs, sa in plan:
                for noprune in ((False, True) if kind == "pfor" and not name.startswith("M") else (False,)):
                    key = f"{name}_{kind}" + ("_noprune" if noprune else "")
                    rec, c = timed(eng, Query(table, sel, ProjectAgg(aggs, ["state"])), sa, noprune)
                    rec["selected_rows"] = int(sum(c[1])) if (c and isinstance(aggs[0], Count)) else None
                    out["records"][key] = rec
                    cols[key] = c
                    print(key, json.dumps(rec), flush=True)
    for name, _, _, _ in plan:
        same = lambda a, b: len(a) == len(b) and all(x.tobytes() == y.tobytes() for x, y in zip(a, b))  # noqa: E731
        out["checks"][f"{name}_pfor_equals_dense"] = same(cols[f"{name}_pfor"], cols[f"{name}_dense"])
        if f"{name}_pfor_noprune" in cols:
            out["checks"][f"{name}_pruned_equals_unpruned"] = same(cols[f"{name}_pfor"], cols[f"{name}_pfor_noprune"])
    if not args.no_oracle:
        with O.Oracle(d_p) as orc:
            exp = orc.query_agg(t_p, oracle_preds(win(10)), [(O.AGG_COUNT, "id"), (O.AGG_MIN, "age"), (O.AGG_MAX, "age")], ["state"],
                                nthreads=os.cpu_count() or 1)
        out["checks"]["W10_pfor_oracle_equal"] = all(np.array_equal(a, b) for a, b in zip(cols["W10_pfor"], exp.columns))
    r = out["records"]
    out["pfor_over_dense_device_median"] = {name: r[f"{name}_pfor"]["device_ms"]["median"] / r[f"{name}_dense"]["device_ms"]["median"]
                                            for name, _, _, _ in plan}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "checks", "pfor_over_dense_device_median")}))
    return 0 if all(out["checks"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
