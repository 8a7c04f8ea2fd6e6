"""The restatement in tests/agg_order_ref.py against the kernel source and the oracle, without a GPU.

The adversarial aggregation tests (tests/test_gpu_agg_order_keys.py) build their key sets from restated hashes.  If the
kernels' hashes or table limits change, those sets silently stop colliding; this file fails instead: it reads k_agg.cuh and
engine.cu and checks the constants and bounds the sets rely on, then checks that each set has the property it claims.
It also checks the reference group-by against the oracle's query_agg, and the canonical-order writer helper against the
oracle's reading of the segments."""
import os
import re

import numpy as np
import pytest

import agg_order_ref as R
import oracle_lib as O
from immutable3_b200 import Count, Max, Min
from immutable3_b200.loader import SegmentWriter

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "immutable3_b200", "csrc")


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _body(src, signature):
    """Text of the function whose definition starts with `signature`, up to its closing brace at column 0."""
    i = src.index(signature)
    return src[i:src.index("\n}\n", i)]


def test_hash_constants_and_limits_match_the_kernel_source():
    src = _src("k_agg.cuh")
    h32 = _body(src, "__device__ __forceinline__ uint32_t agg_hash32(")
    assert f"(uint32_t)k * 0x{R.HASH32_MUL_LO:08X}u" in h32 and f"(uint32_t)(k >> 32) * 0x{R.HASH32_MUL_HI:08X}u" in h32, h32
    h64 = _body(src, "__device__ __forceinline__ uint32_t agg_hash(")
    assert re.search(r"k \^= k >> 33;\s*k \*= 0x%XULL;\s*k \^= k >> 33;\s*return \(uint32_t\)k;" % R.HASH64_MUL, h64, re.I), h64
    assert f"constexpr int kAggSlots = {R.CTA_SLOTS};" in src
    assert f"constexpr int kAggDictBits = {R.DICT_BITS};" in src
    cta = _body(src, "__device__ __forceinline__ int agg_cta_slot(")
    assert "const uint32_t hh = agg_hash32(key);" in cta
    assert "dict + (hh >> (32 - kAggDictBits))" in cta                                    # the guess cache's index
    assert "h = hh >> 24;" in cta                                                         # the home slot
    assert f"for (int p = 0; p < {R.CTA_PROBES}; p++, h = (h + 1) & (kAggSlots - 1))" in cta
    assert "if (*reinterpret_cast<volatile unsigned long long*>(&keys[h]) == key) return (int)h;" in cta   # the guess, confirmed
    glob = _body(src, "__device__ __forceinline__ int agg_global_slot(")
    assert "uint32_t h = agg_hash(key) & (slots - 1);" in glob
    assert "for (uint32_t p = 0; p < slots; p++, h = (h + 1) & (slots - 1))" in glob
    eng = _src("engine.cu")
    assert f"ap.table_slots = 1u << {R.GLOBAL_SLOTS.bit_length() - 1};" in eng
    assert "if (v >= 64 && (v & (v - 1)) == 0) ap.table_slots = v;" in eng              # IMM3_AGG_SLOTS=64 is honoured
    assert "key_bits + 8 * c.meta.width > 56" in eng                                      # 7 key bytes
    assert "ap.group[g].key_shift = key_bits;" in eng


def _c_hash32(k):
    return ((k & 0xFFFFFFFF) * R.HASH32_MUL_LO & 0xFFFFFFFF) ^ (((k >> 32) & 0xFFFFFFFF) * R.HASH32_MUL_HI & 0xFFFFFFFF)


def _c_hash64(k):
    m = (1 << 64) - 1
    k ^= k >> 33
    k = (k * R.HASH64_MUL) & m
    k ^= k >> 33
    return k & 0xFFFFFFFF


def test_vectorised_hashes_equal_the_scalar_statement():
    rng = np.random.default_rng(3)
    keys = np.concatenate([rng.integers(0, 1 << 56, 2000, dtype=np.uint64), np.array([0, 1, (1 << 56) - 1, 0xFFFFFFFF, 1 << 32], np.uint64)])
    h32, h64 = R.agg_hash32(keys), R.agg_hash(keys)
    for i, k in enumerate(keys.tolist()):
        assert int(h32[i]) == _c_hash32(k) and int(h64[i]) == _c_hash64(k), k
    assert (R.cta_home(keys) == h32 >> np.uint64(24)).all() and (R.guess_index(keys) == h32 >> np.uint64(18)).all()


def test_key_packing():
    s3 = np.array([b"\x01\x02\x03", b"\x00\x00\x00", b"\xff\xff\xff"], "S3")
    k = np.array([0x04050607, 0, -1], np.int32)
    b = np.array([-1, 0, 5], np.int8)
    assert R.pack_keys([s3, k]).tolist() == [0x04050607030201, 0, 0x00FFFFFFFFFFFFFF]
    assert R.pack_keys([k, s3]).tolist() == [0x03020104050607, 0, 0x00FFFFFFFFFFFFFF]
    assert R.pack_keys([b, s3]).tolist() == [0x030201FF, 0, 0xFFFFFF05]
    s7 = np.array([b"\x00" * 7, b"\xff" * 7, b"a\x00\x00\x00\x00\x00b"], "S7")
    assert R.pack_keys([s7]).tolist() == [0, 0x00FFFFFFFFFFFFFF, (0x62 << 48) | 0x61]
    assert R.int_keys(k).tolist() == [0x04050607, 0, 0xFFFFFFFF]


def test_adversarial_key_sets_have_their_properties():
    s = R.adversarial_keys()
    hot, cta = s["hot"], s["cta"]
    assert len(set(hot.tolist())) == len(hot) >= R.CTA_PROBES + 1
    assert (R.cta_home(R.int_keys(hot)) == R.CTA_HOME).all()                              # more keys at one home than it probes
    assert len(set(cta.tolist())) == len(cta) < R.SMALL_SLOTS
    g4 = R.int_keys(s["guess4"])
    assert len(set(s["guess4"].tolist())) == 6 and len(set(R.guess_index(g4).tolist())) == 1
    pk = R.pack_keys([s["pair_k"], s["pair_s"]])
    assert len(set(pk.tolist())) == len(pk) and (pk < (1 << 56)).all()
    same = pk[:6]
    assert len(set((same & np.uint64(0xFFFFFFFF)).tolist())) == 1                        # equal low 32 bits ...
    assert len(set(R.guess_index(same).tolist())) == 1                                    # ... and one guess-cache entry
    assert len(set(R.guess_index(pk[6:12]).tolist())) == 1                                # the guess4 keys, 7 bytes wide
    assert (s["pair_s"][6:12].view(np.uint8) == 0).all()
    f64, o65 = s["full64"], s["over65"]
    assert len(set(f64.tolist())) == R.SMALL_SLOTS and len(set(o65.tolist())) == R.SMALL_SLOTS + 1
    assert (R.global_home(R.int_keys(f64), R.SMALL_SLOTS) == R.WRAP_HOME).all()
    assert 0 < R.WRAP_HOME < R.SMALL_SLOTS                                                # filling the table wraps past its last slot
    # the hot keys, introduced over time, then every 1024-row span holds more than 16 of them
    rng = np.random.default_rng(0)
    idx = R.introduced_over_time(cta, 1 << 16, rng)
    first = [int(np.argmax(idx == j)) for j in range(len(cta))]
    assert first == [j * 64 for j in range(len(cta))]
    spans = idx[8192:].reshape(-1, 1024)
    assert min(len(set(r.tolist()) & set(range(len(hot)))) for r in spans) >= R.CTA_PROBES + 1


def test_canonical_segment_order():
    assert R.canonical_segment_order(12) == [0, 1, 10, 11, 2, 3, 4, 5, 6, 7, 8, 9]
    assert R.canonical_segment_order(3) == [0, 1, 2]


@pytest.fixture(scope="module")
def table(tmp_path_factory):
    """13 segments (canonical order != write order) with STRING(1 / 3 / 5 / 7), INT and TINYINT cells, all-0x00 and all-0xFF
    cells among them, written through write_order."""
    d = tmp_path_factory.mktemp("agg_hash_host")
    rng = np.random.default_rng(8)
    n, block, seg = 13 * (4 * 32 + 1) - 40, 32, 4
    cells = lambda w, m: np.array([b"\x00" * w, b"\xff" * w] + [bytes(rng.integers(0, 256, w, dtype=np.uint8)) for _ in range(m)], f"S{w}")
    cols = {"s1": cells(1, 5)[rng.integers(0, 7, n)], "s3": cells(3, 6)[rng.integers(0, 8, n)],
            "s5": cells(5, 9)[rng.integers(0, 11, n)], "s7": cells(7, 9)[rng.integers(0, 11, n)],
            "k": np.array([0, -1, 7, -2**31, 2**31 - 1], np.int32)[rng.integers(0, 5, n)],
            "b": rng.integers(-128, 128, n, dtype=np.int64).astype(np.int8)}
    cols["v"] = rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32)
    specs = ["s1:DENSE_STRING:size=1", "s3:DENSE_STRING:size=3", "s5:DENSE_STRING:size=5", "s7:DENSE_STRING:size=7", "k:DENSE_INT",
             "b:DENSE_TINYINT", "v:DENSE_INT"]
    w = R.write_order(cols, n, block, seg)
    with SegmentWriter(d, "t", specs, block, seg) as wr:
        wr.append(*[w[s.split(":")[0]] for s in specs])
    with O.Oracle(d) as orc:
        yield orc, cols


def test_write_order_puts_the_rows_in_canonical_order(table):
    orc, cols = table
    assert orc.nsegments("t") == 13 and orc.segment_file_ids("t") == R.canonical_segment_order(13)
    names = list(cols)
    got = orc.query("t", [], names)
    for i, c in enumerate(names):
        assert got.columns[i].tobytes() == cols[c].tobytes(), c


@pytest.mark.parametrize("group_by", [["s1"], ["s3"], ["s5"], ["s7"], ["s3", "k"], ["k", "s3"], ["s5", "s1"], ["b", "s5"], ["k"], []])
def test_reference_group_by_equals_the_oracle(table, group_by):
    orc, cols = table
    aggs = [Count("v"), Min("v"), Max("v"), Min("b"), Max("b")]
    ops = {Count: O.AGG_COUNT, Min: O.AGG_MIN, Max: O.AGG_MAX}
    for sel, mask in (([], np.ones(len(cols["v"]), bool)), ([("b", O.OP_GT, -50)], cols["b"] > -50)):
        exp = orc.query_agg("t", sel, [(ops[type(a)], a.col) for a in aggs], group_by)
        got = R.group_by([cols[g][mask] for g in group_by], {c: cols[c][mask] for c in ("v", "b")}, aggs)
        assert len(got) == len(exp.columns)
        for c in range(len(got)):
            assert got[c].dtype == exp.columns[c].dtype and got[c].tobytes() == exp.columns[c].tobytes(), (group_by, c)
