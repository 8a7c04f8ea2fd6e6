"""The IMM3_* experiment switches tests set are real: each one is read somewhere, and every switch DESIGN §4.7 documents is
read by the library.  A switch nobody reads makes a test that sets it run the default configuration again under another
name.  Source scan only: runs without a GPU."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME = r"IMM3_[A-Z0-9_]+"


def _files(rel, exts):
    base = os.path.join(ROOT, rel)
    if os.path.isfile(base):
        yield base
        return
    for dirpath, _, files in os.walk(base):
        for f in sorted(files):
            if f.endswith(exts):
                yield os.path.join(dirpath, f)


def _text(paths):
    return {p: open(p, errors="replace").read() for p in paths}


def _native_reads():
    out = set()
    for src in _text(_files("immutable3_b200/csrc", (".cu", ".cuh", ".cpp", ".hpp", ".h"))).values():
        out |= set(re.findall(rf'getenv\(\s*"({NAME})"\s*\)', src))
    return out


def _python_reads(rels):
    pats = [rf'os\.environ\.get\(\s*["\']({NAME})["\']', rf'os\.getenv\(\s*["\']({NAME})["\']',
            rf'["\']({NAME})["\']\s+(?:not\s+)?in\s+os\.environ', rf'os\.environ\[\s*["\']({NAME})["\']\s*\](?!\s*=[^=])']
    out = set()
    for rel in rels:
        for src in _text(_files(rel, (".py",))).values():
            for p in pats:
                out |= set(re.findall(p, src))
    return out


def _test_sets():
    """IMM3_* names the tests set: monkeypatch.setenv, os.environ[...] = ..., and the keys of environment dicts."""
    pats = [rf'setenv\(\s*["\']({NAME})["\']', rf'os\.environ\[\s*["\']({NAME})["\']\s*\]\s*=[^=]', rf'["\']({NAME})["\']\s*:\s*["\']']
    out = {}
    for path, src in _text(_files("tests", (".py",))).items():
        if os.path.basename(path) == os.path.basename(__file__):
            continue
        for p in pats:
            for n in re.findall(p, src):
                out.setdefault(n, os.path.relpath(path, ROOT))
    return out


def _design_switches():
    txt = open(os.path.join(ROOT, "DESIGN.md")).read()
    m = re.search(r"^### 4\.7 [^\n]*\n(.*?)^#", txt, flags=re.S | re.M)
    assert m, "DESIGN.md has no section 4.7"
    return set(re.findall(NAME, m.group(1)))


def test_every_switch_a_test_sets_is_read():
    reads = _native_reads() | _python_reads(["immutable3_b200", "bench.py", "tools", "tests"])
    sets = _test_sets()
    assert len(sets) >= 10
    dead = {n: where for n, where in sets.items() if n not in reads}
    assert not dead, f"switches set by tests but read nowhere: {dead}"


def test_every_documented_switch_is_read_by_the_library():
    switches = _design_switches()
    assert {"IMM3_NO_LANE", "IMM3_FILTER_STAGES", "IMM3_EMIT_STAGES", "IMM3_PATH"} <= switches
    library = _native_reads() | _python_reads(["immutable3_b200"])
    bench = _python_reads(["bench.py"])
    # (IMM3_BENCH_* switches steer the benchmark script, not the library)
    missing = sorted(n for n in switches if n not in library and not (n.startswith("IMM3_BENCH_") and n in bench))
    assert not missing, f"DESIGN §4.7 lists switches the library never reads: {missing}"
