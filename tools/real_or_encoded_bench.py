"""Real OR over the sorted-int-codec id (imm3_query_begin_dnf_ext with IMM3_DNF_ENCODED_FILTER: every term's block filter front,
merged in block space by blocks_or_merge_kernel) against the same disjunctions on the dense-id twin, which run the row-space
filter kernel once per term (imm3_query_begin_dnf).

  C4         select id from test_1b where id > L and id < H, one 1 % window (imm3_query_begin, for reference)
  O2_0.5     two 0.5 % windows                       O2_5   two 5 % windows
  O4         four 0.5 % windows                      OWS    a 1 % window or (state = 'CA' and age = 7)
bench.py's tables (1 B rows by default) and the protocol of tools/agg_encoded_filter_bench.py: >= 3 warm-up and >= 20 timed
steps per query, the L2 evicted by a 512 MiB read pass before each, median and min of the CUDA-event time of the query's kernels
(Result.device_ms) and of the wall time of Engine.begin (kernels + match count, no row read-back).  Check: every query's rows
equal on the encoded table and the dense twin.  The GPU's name and power limit are read in the same run.

usage: python tools/real_or_encoded_bench.py [--rows N] [--steps K] [--warmup W] [--out profiles/<name>.json]"""
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_real_or_encoded.json"))
    args = ap.parse_args()
    args.steps, args.warmup = max(20, args.steps), max(3, args.warmup)

    import numpy as np
    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the filter kernels have no CPU fallback"}))
        return 2
    from helpers import conj
    from immutable3_b200 import EQ, GT, LT, And, Engine, Match, Max, Min, NoSelect, Or, Project, ProjectAgg, Query, SegmentManager, Select

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    flush_buf = torch.zeros(512 << 20, dtype=torch.uint8, device="cuda")
    flush_sink = torch.zeros((), dtype=torch.int64, device="cuda")

    def flush_l2():
        flush_sink.copy_(flush_buf.view(torch.int64).sum())
        torch.cuda.synchronize()

    def timed(eng, q, real_or, encoded):
        wall, dev = [], []
        for i in range(args.warmup + args.steps):
            flush_l2()
            t0 = time.perf_counter()
            r = eng.begin(q, real_or=real_or, encoded_filter=encoded) if real_or else eng.begin(q)
            t1 = time.perf_counter()
            if i >= args.warmup:
                wall.append((t1 - t0) * 1e3)
                dev.append(r.device_ms)
            if i == args.warmup + args.steps - 1:
                r.fetch(r.take)
                col, route, alg = np.asarray(r.column(0)), r.route, r.algorithmic_bytes
            r.close()
        rec = {"rows": int(len(col)), "route": route, "algorithmic_bytes": alg,
               "device_ms": {"median": statistics.median(dev), "min": min(dev)}, "wall_ms": {"median": statistics.median(wall), "min": min(wall)}}
        return rec, col

    out = {"gpu": gpu, "rows": args.rows, "steps": args.steps, "warmup": args.warmup,
           "protocol": "per step: 512 MiB read pass (L2 eviction), then Engine.begin(..., real_or=True[, encoded_filter=True]); device = CUDA "
                       "events around the query's kernels; wall = Engine.begin (no row read-back)",
           "queries": {"C4": "select id from test_1b where id > L and id < H (1 % window, imm3_query_begin)",
                       "O2_0.5": "two 0.5 % windows", "O2_5": "two 5 % windows", "O4": "four 0.5 % windows",
                       "OWS": "a 1 % window or (state = 'CA' and age = 7)"},
           "windows": {}, "checks": {}, "records": {}}
    d_p, t_p, _ = bench.ensure_table("pfor", args.rows, 0, 1, lambda: None, "product")
    d_d, t_d, _ = bench.ensure_table("dense", args.rows, 0, 1, lambda: None, "product")
    with SegmentManager(d_p) as sm:
        with Engine(sm).execute(Query(t_p, NoSelect, ProjectAgg([Min("id"), Max("id")], []))) as r:
            lo, hi = int(r.column(0)[0]), int(r.column(1)[0])

    def win(at, pct):  # about pct % of the ids, starting at fraction `at` of the id range
        a = lo + int((hi - lo) * at)
        out["windows"][f"{at}:{pct}"] = [a, a + int((hi - lo) * pct / 100)]
        return conj(Select("id", GT(a)), Select("id", LT(a + int((hi - lo) * pct / 100))))

    plan = [("C4", win(0.495, 1), False),
            ("O2_0.5", Or(win(0.2, 0.5), win(0.7, 0.5)), True),
            ("O2_5", Or(win(0.1, 5), win(0.6, 5)), True),
            ("O4", Or(Or(win(0.1, 0.5), win(0.35, 0.5)), Or(win(0.6, 0.5), win(0.85, 0.5))), True),
            ("OWS", Or(win(0.495, 1), And(Select("state", Match(["CA"])), Select("age", EQ(7)))), True)]
    cols = {}
    for kind, d, table in (("pfor", d_p, t_p), ("dense", d_d, t_d)):
        with SegmentManager(d) as sm:
            eng = Engine(sm)
            for name, sel, real_or in plan:
                key = f"{name}_{kind}"
                rec, c = timed(eng, Query(table, sel, Project(["id"])), real_or, kind == "pfor")
                out["records"][key] = rec
                cols[key] = c
                print(key, json.dumps(rec), flush=True)
    for name, _, _ in plan:
        out["checks"][f"{name}_pfor_equals_dense"] = cols[f"{name}_pfor"].tobytes() == cols[f"{name}_dense"].tobytes()
    r = out["records"]
    out["pfor_over_dense_device_median"] = {name: r[f"{name}_pfor"]["device_ms"]["median"] / r[f"{name}_dense"]["device_ms"]["median"]
                                            for name, _, _ in plan}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "checks", "pfor_over_dense_device_median")}))
    return 0 if all(out["checks"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
