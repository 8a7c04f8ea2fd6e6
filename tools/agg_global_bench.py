"""Global aggregates across segment-sharded GPUs: imm3_query_agg (this rank's partials) against imm3_query_agg_global
(partials merged on the GPUs over NVLink) and against partials + a host merge over a gloo all_gather_object.

Workloads (bench.py's synthetic tables, written once and reused):
  example  select min(age), max(age) from T where age > 18 group by state - the reference's example (Engine.scala:66-78),
           weak scaling: 100 M rows per rank on the dense-id table
  q1       select count(id), min(id), max(id) from T where age > 18 group by state - Q1 of tools/agg_encoded_bench.py,
           strong scaling on test_1b (id in the sorted-int codec, 1 B rows)
Per step: a 512 MiB read pass evicts the L2, then the query; >= 3 warm-up and >= 20 timed steps per arm, median and min.
device = CUDA-event time of the query's kernels (Result.device_ms; for the global form it spans through the merge), wall =
host time around the call (for the host-merge arm: partials + all_gather_object + merge_partials).  Rank 0 checks the global
result against the oracle over the whole table once per configuration and writes profiles/r4_agg_global_n{N}.json with the
GPU's name and power limit read in the same run.

usage: python -m torch.distributed.run --nproc_per_node N tools/agg_global_bench.py [--workloads example,q1] [--steps K]"""
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

WORKLOADS = {
    "example": ("select min(age), max(age) from T where age > 18 group by state", "dense", 100_000_000, True,
                [("age", 1, 18)], [(1, "age"), (2, "age")], ["state"]),
    "q1": ("select count(id), min(id), max(id) from T where age > 18 group by state", "pfor", 1_000_000_000, False,
           [("age", 1, 18)], [(0, "id"), (1, "id"), (2, "id")], ["state"]),
}


def build_query(table, preds, aggs, group_by):
    from immutable3_b200 import GT, And, Count, Max, Min, NoSelect, ProjectAgg, Query, Select

    sel = NoSelect
    for i, (c, _, v) in enumerate(preds):
        sel = Select(c, GT(v)) if i == 0 else And(sel, Select(c, GT(v)))
    return Query(table, sel, ProjectAgg([{0: Count, 1: Min, 2: Max}[op](col) for op, col in aggs], group_by))


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="example,q1")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rows-per-rank", type=int, default=0, help="override the weak workload's rows per rank")
    ap.add_argument("--rows", type=int, default=0, help="override the strong workload's rows")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    args.steps, args.warmup = max(20, args.steps), max(3, args.warmup)

    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the aggregation kernels have no CPU fallback"}))
        return 2
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    ndev = torch.cuda.device_count()
    if world > ndev:
        print(json.dumps({"error": f"{world} ranks on {ndev} GPU(s): one GPU per rank is measured, not ranks sharing a GPU"}))
        return 2
    torch.cuda.set_device(rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))  # (torch.distributed.run's environment)
    else:
        dist.init_process_group("gloo")
    host_group = dist.new_group(backend="gloo")  # the host merge's channel
    barrier = lambda: dist.barrier(group=host_group)  # noqa: E731
    import oracle_lib as O
    from immutable3_b200 import Engine, SegmentManager
    from immutable3_b200.dist import merge_partials

    gpu = subprocess.run(["nvidia-smi", "-i", str(rank), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    flush_buf = torch.zeros(512 << 20, dtype=torch.uint8, device="cuda")
    flush_sink = torch.zeros((), dtype=torch.int64, device="cuda")

    def flush_l2():
        flush_sink.copy_(flush_buf.view(torch.int64).sum())
        torch.cuda.synchronize()

    out = {"gpu": gpu, "world": world, "steps": args.steps, "warmup": args.warmup,
           "protocol": "per step: 512 MiB read pass (L2 eviction), then the call; device = CUDA events around the query's kernels",
           "workloads": {}}
    for name in [w for w in args.workloads.split(",") if w]:
        what, kind, rows, weak, preds, aggs, group_by = WORKLOADS[name]
        if weak:
            rows = (args.rows_per_rank or rows) * world
        elif args.rows:
            rows = args.rows
        if rank == 0:
            print(f"{name}: preparing {rows} rows", flush=True)
        d, table, _ = bench.ensure_table(kind, rows, rank, world, barrier, "product")
        q = build_query(table, preds, aggs, group_by)
        sm = SegmentManager(d, device=rank, rank=rank, world=world)
        sm.comm_connect()
        eng = Engine(sm)

        def partial():
            return eng.execute(q)

        def global_():
            return eng.execute_agg_global(q)

        def host_merge():
            r = eng.execute(q)
            everyone = [None] * world
            dist.all_gather_object(everyone, r.columns(), group=host_group)
            return r, merge_partials(everyone, len(group_by), list(q.project.aggs))

        rec = {"what": what, "table": table, "rows": rows, "scaling": "weak" if weak else "strong"}
        last = {}
        for arm, fn in (("partials", partial), ("global", global_), ("partials_host_merge", host_merge)):
            wall, dev = [], []
            for i in range(args.warmup + args.steps):
                flush_l2()
                barrier()
                t0 = time.perf_counter()
                got = fn()
                t1 = time.perf_counter()
                r, cols = got if isinstance(got, tuple) else (got, None)
                if i >= args.warmup:
                    wall.append((t1 - t0) * 1e3)
                    dev.append(r.device_ms)
                if i == args.warmup + args.steps - 1:
                    last[arm] = cols if cols is not None else [np.asarray(c) for c in r.columns()]
                    if arm == "global":
                        rec["route"] = r.route
                        rec["groups"] = r.global_count
                        rec["rank_partial_groups"] = r.rank_counts
                r.close()
            rec[arm] = {"device_ms": summary(dev), "wall_ms": summary(wall)}
            if rank == 0:
                print(f"{name} {arm}: {json.dumps(rec[arm])}", flush=True)
        rec["host_merge_equal"] = len(last["global"]) == len(last["partials_host_merge"]) and all(
            np.array_equal(a, b) for a, b in zip(last["global"], last["partials_host_merge"]))
        if rank == 0:
            with O.Oracle(d) as orc:
                exp = orc.query_agg(table, preds, aggs, group_by, nthreads=os.cpu_count() or 1)
            rec["oracle_equal"] = len(last["global"]) == len(exp.columns) and all(np.array_equal(a, np.asarray(b)) for a, b in zip(last["global"], exp.columns))
        # every rank's timings: the query ends when the slowest rank's does
        per_rank = [None] * world
        dist.all_gather_object(per_rank, {arm: rec[arm] for arm in ("partials", "global", "partials_host_merge")}, group=host_group)
        rec["per_rank"] = per_rank
        out["workloads"][name] = rec
        if rank == 0:
            print(name, json.dumps({k: rec[k] for k in ("partials", "global", "partials_host_merge", "oracle_equal", "host_merge_equal")}), flush=True)
        sm.close()
        barrier()
    if rank == 0:
        path = args.out or os.path.join(ROOT, "profiles", f"r4_agg_global_n{world}.json")
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            json.dump(out, f, indent=1)
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
