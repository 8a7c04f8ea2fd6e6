"""bench.py's reference arm (the CPU restatement of the reference path, SURVEY.md 8d) prints the contract's JSON line; its `config`
is built by the same function as the GPU arm's, so the two lines describe one configuration.  Both arms write the result of their
last timed step with --dump-outputs; the GPU arm's test needs a B200."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    env = dict(os.environ, IMM3_BENCH_ALLOW_SHORT="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def _load_dump(d):
    return {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_reference_arm_prints_the_contract_line(tmp_path):
    line = _bench("--impl", "reference", "--rows", "2100000", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path / "out"))
    assert line["impl"] == "reference" and line["metric"] == "rows/sec for scan+filter+project" and line["unit"] == "rows/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cfg = line["config"]
    assert cfg["rows_total"] == 2100000 and cfg["segments"] == 3 and cfg["scaling"] == "strong" and "C4" in cfg["workload"]
    assert cfg["result_rows"] == line["result_rows"] == 20999          # the 1 % id window, both ends exclusive
    dump = _load_dump(tmp_path / "out")
    assert sorted(dump) == ["id.npy", "result_rows.npy"]
    assert dump["id.npy"].dtype == np.float64 and np.array_equal(dump["id.npy"], np.arange(1039501, 1060500))  # synthetic id = row index
    assert dump["result_rows.npy"].tolist() == [20999]


def test_dump_outputs_samples_a_large_result_the_same_way_every_time(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 64 << 10)
    n = 50_000
    ids = np.arange(n, dtype=np.int32) * 7
    states = np.array([b"CA", b"NY", b"TX"], dtype="S2")[np.arange(n) % 3]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ["id", "state"], [ids, states], n)
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    assert sorted(a) == ["id.npy", "result_rows.npy", "sample_rows.npy", "state.npy"]
    assert all(np.array_equal(a[f], b[f]) for f in a)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in a) <= 64 << 10
    rows = a["sample_rows.npy"].astype(np.int64)
    assert len(rows) > 1000 and np.all(np.diff(rows) > 0) and rows[-1] < n
    assert np.array_equal(a["id.npy"], ids[rows]) and a["result_rows.npy"].tolist() == [n]
    assert a["state.npy"].shape == (len(rows), 2) and np.array_equal(a["state.npy"].astype(np.uint8).view("S2").ravel(), states[rows])


def test_both_arms_build_config_from_the_same_function():
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count("protocol_keys(args,") == 3                       # the definition, reference_arm and the GPU arm
    assert src.count('"config": config_dict(args, args.workload, total, world, protocol_keys(') == 2


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["c4", "c3", "agg"])
def test_gpu_arm_dumps_what_the_reference_arm_computes(tmp_path, workload):
    common = ["--workload", workload, "--rows", "2100000"]
    line = _bench(*common, "--steps", "2", "--warmup", "3", "--no-e2e", "--no-secondary", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "gpu"))
    assert line["steps"] == 2 and line["result_equal"] == [True]
    _bench("--impl", "reference", *common, "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "ref"))
    gpu, ref = _load_dump(tmp_path / "gpu"), _load_dump(tmp_path / "ref")
    assert sorted(gpu) == sorted(ref) and "result_rows.npy" in gpu and len(gpu) >= 2
    for f in gpu:
        assert gpu[f].dtype == np.float64 and np.array_equal(gpu[f], ref[f]), f
    assert gpu["result_rows.npy"].tolist() == [line["config"]["result_rows"]]
