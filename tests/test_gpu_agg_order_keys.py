"""Group order and group keys where the aggregation kernels loop, pack and collide (k_agg.cuh), against an exact numpy
group-by (agg_order_ref.py) and the oracle.

Results come back in the order in which groups first appear in canonical row order; the host sorts the groups by the first
row the kernels' fold rebuilds from a warp's ordinal.  This file checks the parts of that shared code the other aggregate
tests cannot reach:
  A  first rows rebuilt once a warp loops: 24 M rows, groups introduced over time (and single-row groups placed late), so
     that groups first appear after several grid strides - agg_kernel with and without SUM, agg_blocks_kernel, and the
     block-space selection (/bsel);
  B  group cells of every width, gathered byte by byte when they are not 1, 2 or 4 bytes wide, packed into 7-byte keys, with
     all-0x00 and all-0xFF cells (key 0 and 0x00FF..FF), on blocks whose first row is not a multiple of 4;
  C  key sets constructed from the restated hashes: more keys at one CTA home than agg_cta_slot probes, keys sharing a
     guess-cache entry (7-byte keys with equal low 32 bits among them), and a 64-slot global table filled exactly, its
     probe sequence wrapping past the last slot (65 groups: refused);
  D  the global merge when the ranks' first-appearance orders disagree, at 2 and 3 ranks, device and host exchange."""
import os
import sys
import time

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import agg_order_ref as R
import oracle_lib as O
from agg_sum_ref import query_agg_ext
from helpers import conj, oracle_preds
from immutable3_b200 import Avg, Count, Engine, GT, Imm3Error, LT, Max, Min, NoSelect, ProjectAgg, Query, SegmentManager, Select, Sum
from immutable3_b200 import _lib as L
from immutable3_b200.loader import SegmentWriter

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
I32_MIN, I32_MAX = -2**31, 2**31 - 1
_OPS = {Count: O.AGG_COUNT, Min: O.AGG_MIN, Max: O.AGG_MAX}


def write_table(d, name, cols, specs, block, seg):
    """Columns given in CANONICAL order (name -> array; a twin column names the same array) -> segments."""
    names = [s.split(":")[0] for s in specs]
    n = len(cols[names[0]])
    w = R.write_order({c: cols[c] for c in names}, n, block, seg)
    with SegmentWriter(d, name, specs, block, seg) as wr:
        for a in range(0, n, 1 << 21):
            wr.append(*[w[c][a:a + (1 << 21)] for c in names])


def _first_diff(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if len(a) != len(b):
        return f"lengths {len(a)} / {len(b)}"
    bad = np.flatnonzero((a.view(np.uint8).reshape(len(a), -1) != b.view(np.uint8).reshape(len(b), -1)).any(axis=1))
    return f"first difference at group {bad[0]} of {len(a)}: {a[bad[0]]!r} / {b[bad[0]]!r}" if len(bad) else "equal"


def check(eng, table, sel, aggs, gb, exp, kern, **kw):
    """The query on the GPU against the expected columns (group cells, then one per aggregate), compared as raw bytes;
    `kern` = the aggregation kernel the route must show.  Returns the number of groups."""
    with eng.execute(Query(table, sel, ProjectAgg(aggs, gb)), **kw) as got:
        r = got.route
        assert f";{kern};agg_compact" in r, (kern, r)
        assert got.kernel_launches == len(r.split(";")), (got.kernel_launches, r)
        n = len(exp[0])
        assert got.nrows == n and got.ncols == len(gb) + len(aggs), (table, sel, aggs, gb, got.nrows, n, r)
        for c in range(got.ncols):
            g = got.column(c)
            e = np.asarray(exp[c]).astype(g.dtype)
            assert g.tobytes() == e.tobytes(), (table, sel, aggs, gb, c, r, _first_diff(g, e))
        return n


# ---- A. late first rows at scale ------------------------------------------------------------------------------------------

A_ROWS, A_BLOCK, A_SEG = 24_000_000, 1024, 1000
A_GROUPS = (200, 5000, 60000)
A_LATE = (0.41, 0.63, 0.87, 0.995)          # single-row groups at these fractions of the table


def _window_a(n):
    return conj(Select("w", GT(int(n * 0.05))), Select("w", LT(int(n * 0.97))))


@pytest.fixture(scope="module")
def late(tmp_path_factory):
    """24 M rows, 24 segments: per G a group column g<G> whose row i draws uniformly from the first 1 + G * i / n keys of a
    random permutation (and 4 single-row groups placed late), its TINYINT function h<G>, its PFOR_INT twin p<G>; full-range
    INT v (and its PFOR_INT twin vp) and TINYINT t; w = the canonical row number, PFOR_INT (the window of the block filter)."""
    d = tmp_path_factory.mktemp("agg_late")
    t0 = time.time()
    rng = np.random.default_rng(2024)
    n = A_ROWS
    row = np.arange(n, dtype=np.int64)
    cols = {}
    specs = []
    pool = rng.choice(np.arange(I32_MIN, I32_MAX, 4099, dtype=np.int64), 70_000, replace=False).astype(np.int32)
    for G in A_GROUPS:
        keys = pool[:G].copy()
        keys[rng.integers(0, G, 4)] = [0, -1, I32_MIN, I32_MAX]     # (the extremes among the keys, wherever they fall)
        keys = np.unique(keys)
        keys = keys[rng.permutation(len(keys))]
        idx = np.minimum((rng.random(n) * (1 + len(keys) * row / n)).astype(np.int64), len(keys) - 1)
        g = keys[idx]
        g[[int(f * n) for f in A_LATE]] = pool[-1 - np.arange(len(A_LATE))]   # keys found nowhere else
        cols[f"g{G}"] = cols[f"p{G}"] = g
        cols[f"h{G}"] = ((g.view(np.uint32).astype(np.uint64) * np.uint64(R.HASH32_MUL_LO)) >> np.uint64(24)).astype(np.uint8).view(np.int8)
        specs += [f"g{G}:DENSE_INT", f"h{G}:DENSE_TINYINT", f"p{G}:PFOR_INT"]
    v = rng.integers(I32_MIN, I32_MAX, n, dtype=np.int64, endpoint=True).astype(np.int32)
    v[rng.integers(0, n, 64)] = I32_MIN
    v[rng.integers(0, n, 64)] = I32_MAX
    cols["v"] = cols["vp"] = v
    cols["t"] = rng.integers(-128, 128, n, dtype=np.int64).astype(np.int8)
    cols["w"] = row.astype(np.int32)
    specs += ["v:DENSE_INT", "vp:PFOR_INT", "t:DENSE_TINYINT", "w:PFOR_INT"]
    write_table(d, "late", cols, specs, A_BLOCK, A_SEG)
    with O.Oracle(d) as orc:
        nseg = orc.nsegments("late")
        assert orc.segment_file_ids("late") == R.canonical_segment_order(nseg) != list(range(nseg))
        assert orc.query("late", [], ["t"]).columns[0].tobytes() == cols["t"].tobytes()        # write_order = canonical order
    print(f"\n[late] {n} rows, {nseg} segments written in {time.time() - t0:.1f} s")
    sm = SegmentManager(d)
    yield sm, cols
    sm.close()


def _premise_a(groups, G):
    """Loop depth: more 1024-row spans (and blocks) than 4 x SMs x 4 CTAs x 8 warps, so that every warp of a grid of at most
    4 aggregation CTAs per SM (each needs ~50 KB of shared memory) passes at least 4 spans; and many groups first appear
    beyond the first grid stride."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = A_ROWS
    spans = (n + 1023) // 1024
    per = A_BLOCK * A_SEG + 1
    blocks = sum((min(per, n - s * per) + A_BLOCK - 1) // A_BLOCK for s in range((n + per - 1) // per))
    bound = 4 * sms * 4 * 8
    first = groups.first
    stride_rows = sms * 4 * 8 * 1024
    late = int((first >= stride_rows).sum())
    print(f"[late G={G}] SMs {sms}: spans {spans}, blocks {blocks} > 4 x SMs x 4 x 8 = {bound}; {len(first)} groups, "
          f"{late} first appear beyond the first grid stride ({stride_rows} rows), the last at row {int(first[-1])}")
    assert spans > bound and blocks > bound
    assert late >= len(first) // 2 and first[-1] >= int(A_LATE[-1] * n)


@pytest.mark.parametrize("G", A_GROUPS)
def test_late_first_rows(late, G):
    sm, cols = late
    eng = Engine(sm)
    n = A_ROWS
    g, h, p = f"g{G}", f"h{G}", f"p{G}"
    sel_p = Select("t", GT(-120))
    masks = {"all": None, "p": cols["t"] > -120, "w": (cols["w"] > int(n * 0.05)) & (cols["w"] < int(n * 0.97)) & (cols["t"] > -120)}
    cache = {}

    def expect(which, gb, aggs):
        """Expected columns; h<G> is a function of g<G>, so every grouping of this test has the groups of g<G>."""
        m = masks[which]
        if which not in cache:
            key = cols[g] if m is None else cols[g][m]
            cache[which] = R.Groups([key], len(key))
        sub = lambda c: cols[c] if m is None else cols[c][m]
        return R.group_by([sub(c) for c in gb], {c: sub(c) for c in ("v", "vp", "t")}, aggs, groups=cache[which])

    na = {1: [Count("v")],
          3: [Min("v"), Max("v"), Count("v")],
          8: [Min("v"), Max("v"), Count("t"), Min("t"), Max("t"), Max("v"), Min("v"), Count("v")]}
    t0 = time.time()
    expect("all", [g], [])
    _premise_a(cache["all"], G)
    ngroups = None
    for gb, ng in (([g], 1), ([g, h], 2), ([h, g, h], 4)):
        for k, aggs in na.items():
            which, sel = ("all", NoSelect) if k == 1 else ("p", sel_p)
            got = check(eng, "late", sel, aggs, gb, expect(which, gb, aggs), f"agg<{ng},{k}>")
            ngroups = got if which == "all" else ngroups
    aggs = [Sum("v"), Avg("v"), Avg("t"), Min("v"), Max("t")]
    check(eng, "late", sel_p, aggs, [g], expect("p", [g], aggs), "agg<1,8>/sum", sum_avg=True)
    aggs = [Sum("t"), Count("v")]
    check(eng, "late", NoSelect, aggs, [g, h], expect("all", [g, h], aggs), "agg<2,2>/sum", sum_avg=True)
    # agg_blocks_kernel: the PFOR_INT twin as the group column, a PFOR_INT MIN input, SUM
    aggs = [Count("v"), Min("v"), Max("v")]
    check(eng, "late", sel_p, aggs, [p], expect("p", [g], aggs), "agg_blocks<1,3>")
    aggs = [Min("vp"), Max("t")]
    check(eng, "late", sel_p, aggs, [g], expect("p", [g], aggs), "agg_blocks<1,2>")
    aggs = [Sum("v"), Avg("vp")]
    check(eng, "late", NoSelect, aggs, [p], expect("all", [g], aggs), "agg_blocks<1,3>/sum", sum_avg=True)
    # the block-space selection: a window on a PFOR_INT column and a dense predicate
    aggs = [Count("v"), Min("v"), Max("v"), Min("t")]
    check(eng, "late", conj(_window_a(n), sel_p), aggs, [g], expect("w", [g], aggs), "agg_blocks<1,4>/bsel", encoded_filter=True)
    aggs = [Sum("v"), Avg("t")]
    check(eng, "late", conj(_window_a(n), sel_p), aggs, [p], expect("w", [g], aggs), "agg_blocks<1,3>/sum/bsel", sum_avg=True, encoded_filter=True)
    print(f"[late G={G}] {ngroups} groups; 16 queries checked in {time.time() - t0:.1f} s")
    assert ngroups >= 0.9 * G


# ---- B. every key width ---------------------------------------------------------------------------------------------------

B_TABLES = {"kw1000": (50_000, 1000, 4), "kw100": (50_000, 100, 20)}     # 13 and 25 segments
B_GROUPINGS = [["s1"], ["s3"], ["s5"], ["s6"], ["s7"],                     # each width alone
               ["s3", "k"], ["s3", "kp"], ["k", "s3"], ["s5", "s2"], ["s6", "s1"], ["s6", "b"], ["b", "s6"]]   # 7 bytes


@pytest.fixture(scope="module")
def keys_world(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg_keys")
    rng = np.random.default_rng(77)
    tables = {}
    for name, (n, block, seg) in B_TABLES.items():
        def cells(w, m):
            c = [bytes(rng.integers(0, 256, w, dtype=np.uint8)) for _ in range(m)]
            c += [b"\x00" * (w - 1) + b"\x01", b"\x01" + b"\x00" * (w - 1), b"\xff" * (w - 1) + b"\x00"]   # NULs at either end
            return np.array(c, f"S{w}")[rng.integers(0, len(c), n)]
        cols = {f"s{w}": cells(w, 9) for w in (1, 2, 3, 5, 6, 7)}
        cols["k"] = np.array([0, -1, 1, 256, -256, I32_MIN, I32_MAX, 0x00FF00FF], np.int32)[rng.integers(0, 8, n)]
        cols["b"] = np.array([0, -1, 1, -128, 127, 64], np.int8)[rng.integers(0, 6, n)]
        zero, ones = rng.random(n) < 0.02, rng.random(n) < 0.02          # every group cell all-0x00, or all-0xFF
        for w in (1, 2, 3, 5, 6, 7):
            cols[f"s{w}"][zero] = b"\x00" * w
            cols[f"s{w}"][ones & ~zero] = b"\xff" * w
        cols["k"][zero], cols["b"][zero] = 0, 0
        cols["k"][ones & ~zero], cols["b"][ones & ~zero] = -1, -1
        cols["kp"] = cols["k"]
        cols["v"] = cols["vp"] = rng.integers(I32_MIN, I32_MAX, n, dtype=np.int64, endpoint=True).astype(np.int32)
        cols["w"] = np.arange(n, dtype=np.int32)
        specs = [f"s{w}:DENSE_STRING:size={w}" for w in (1, 2, 3, 5, 6, 7)] + ["k:DENSE_INT", "kp:PFOR_INT", "b:DENSE_TINYINT", "v:DENSE_INT",
                                                                            "vp:PFOR_INT", "w:PFOR_INT"]
        write_table(d, name, cols, specs, block, seg)
        tables[name] = cols
    orc, sm = O.Oracle(d), SegmentManager(d)
    for name, cols in tables.items():
        assert orc.nsegments(name) > 10
        got = orc.query(name, [], list(cols))
        for i, c in enumerate(cols):
            assert got.columns[i].tobytes() == cols[c].tobytes(), (name, c)                      # canonical order as meant
    yield orc, sm, tables
    sm.close()
    orc.close()


def _oracle_cols(orc, table, sel, aggs, gb):
    if any(isinstance(a, (Sum, Avg)) for a in aggs):
        return query_agg_ext(orc, table, sel, aggs, gb)
    return orc.query_agg(table, oracle_preds(sel), [(_OPS[type(a)], a.col) for a in aggs], list(gb)).columns


@pytest.mark.parametrize("table", list(B_TABLES))
def test_every_key_width(keys_world, table):
    orc, sm, tables = keys_world
    cols = tables[table]
    eng = Engine(sm)
    n = len(cols["v"])
    sel_p = Select("b", GT(-100))
    win = conj(Select("w", GT(n // 20)), Select("w", LT(n - n // 20)), sel_p)
    masks = {"p": cols["b"] > -100}
    masks["w"] = masks["p"] & (cols["w"] > n // 20) & (cols["w"] < n - n // 20)
    for gb in B_GROUPINGS:
        width = sum(cols[c].dtype.itemsize for c in gb)
        enc = any(c.endswith("p") for c in gb)
        ng = len(gb) if len(gb) <= 2 else 4
        for m in masks.values():                                          # key 0 and 0x00FF..FF occur in every grouping
            keys = set(R.pack_keys([cols[c][m] for c in gb]).tolist())
            assert 0 in keys and (1 << (8 * width)) - 1 in keys, gb
        cases = [(sel_p, [Count("v"), Min("v"), Max("v")], "p", f"agg_blocks<{ng},3>" if enc else f"agg<{ng},3>", {}),
                 (sel_p, [Count("v"), Min("vp"), Max("v")], "p", f"agg_blocks<{ng},3>", {}),
                 (sel_p, [Sum("v"), Avg("v"), Min("b")], "p", f"agg_blocks<{ng},4>/sum" if enc else f"agg<{ng},4>/sum", {"sum_avg": True}),
                 (win, [Count("v"), Min("v"), Max("b")], "w", f"agg_blocks<{ng},3>/bsel", {"encoded_filter": True}),
                 (win, [Sum("v"), Avg("b")], "w", f"agg_blocks<{ng},3>/sum/bsel", {"encoded_filter": True, "sum_avg": True})]
        for sel, aggs, which, kern, kw in cases:
            m = masks[which]
            exp = R.group_by([cols[c][m] for c in gb], {c: cols[c][m] for c in ("v", "vp", "b")}, aggs)
            ref = _oracle_cols(orc, table, sel, aggs, gb)
            assert len(ref) == len(exp)
            for c in range(len(exp)):                                     # the numpy reference is the oracle's answer
                assert np.asarray(ref[c]).astype(exp[c].dtype).tobytes() == exp[c].tobytes(), (table, gb, aggs, c)
            check(eng, table, sel, aggs, gb, exp, kern, **kw)


# ---- C. adversarial keys --------------------------------------------------------------------------------------------------

C_ROWS, C_BLOCK, C_SEG = 1_000_000, 1024, 40                              # 25 segments


@pytest.fixture(scope="module")
def adversarial(tmp_path_factory):
    """c1: the 44 groups of which 24 share a CTA home; c2 (+ s3): the guess-sharing keys and 7-byte pairs; c3: 64 keys of one
    home in a 64-slot table; c4: 65 keys.  Key j of a set first appears at row 64 j, every later row draws uniformly from the
    keys introduced by then.  c<i>p = the PFOR_INT twin of c<i>."""
    d = tmp_path_factory.mktemp("agg_adv")
    rng = np.random.default_rng(99)
    s = R.adversarial_keys()
    n = C_ROWS
    cols = {}
    cols["c1"] = cols["c1p"] = s["cta"][R.introduced_over_time(s["cta"], n, rng)]
    pi = R.introduced_over_time(s["pair_k"], n, rng)
    cols["c2"] = cols["c2p"] = s["pair_k"][pi]
    cols["s3"] = s["pair_s"][pi]
    cols["c3"] = cols["c3p"] = s["full64"][R.introduced_over_time(s["full64"], n, rng)]
    cols["c4"] = cols["c4p"] = s["over65"][R.introduced_over_time(s["over65"], n, rng)]
    cols["v"] = rng.integers(I32_MIN, I32_MAX, n, dtype=np.int64, endpoint=True).astype(np.int32)
    cols["b"] = rng.integers(-128, 128, n, dtype=np.int64).astype(np.int8)
    specs = ["c1:DENSE_INT", "c1p:PFOR_INT", "c2:DENSE_INT", "c2p:PFOR_INT", "s3:DENSE_STRING:size=3", "c3:DENSE_INT", "c3p:PFOR_INT",
             "c4:DENSE_INT", "c4p:PFOR_INT", "v:DENSE_INT", "b:DENSE_TINYINT"]
    write_table(d, "adv", cols, specs, C_BLOCK, C_SEG)
    # premise: every 1024-row span (so every warp's first span, and every CTA) holds more of the hot keys than a CTA probes
    hot = np.isin(cols["c1"], s["hot"])
    per_span = [len(np.unique(cols["c1"][a:a + 1024][hot[a:a + 1024]])) for a in range(1024, n - 1024, 1024)]
    print(f"\n[adversarial] {len(s['hot'])} of {len(s['cta'])} keys at CTA home {R.CTA_HOME}; every span past the first holds "
          f">= {min(per_span)} of them; 64 keys at global home {R.WRAP_HOME} of {R.SMALL_SLOTS}")
    assert min(per_span) >= R.CTA_PROBES + 1
    orc, sm = O.Oracle(d), SegmentManager(d)
    assert orc.nsegments("adv") > 10
    yield orc, sm, cols
    sm.close()
    orc.close()


def _check_c(orc, eng, cols, sel, mask, aggs, gb, kern, **kw):
    exp = R.group_by([cols[c][mask] for c in gb], {c: cols[c][mask] for c in ("v", "b")}, aggs)
    ref = _oracle_cols(orc, "adv", sel, aggs, gb)
    for c in range(len(exp)):
        assert np.asarray(ref[c]).astype(exp[c].dtype).tobytes() == exp[c].tobytes(), (gb, aggs, c)
    return check(eng, "adv", sel, aggs, gb, exp, kern, **kw)


@pytest.mark.parametrize("enc", [False, True], ids=["dense", "encoded"])
@pytest.mark.parametrize("with_sum", [False, True], ids=["count_min_max", "sum"])
def test_adversarial_keys(adversarial, monkeypatch, enc, with_sum):
    orc, sm, cols = adversarial
    eng = Engine(sm)
    n = C_ROWS
    kname = "agg_blocks" if enc else "agg"
    col = lambda i: f"c{i}p" if enc else f"c{i}"
    sel, mask = Select("b", GT(-120)), cols["b"] > -120
    aggs = [Sum("v"), Avg("b"), Min("v"), Count("v")] if with_sum else [Count("v"), Min("v"), Max("v"), Max("b")]
    kw = {"sum_avg": True} if with_sum else {}
    sfx = "/sum" if with_sum else ""
    every = np.ones(n, bool)
    for s_, m_ in ((NoSelect, every), (sel, mask)):
        assert _check_c(orc, eng, cols, s_, m_, aggs, [col(1)], f"{kname}<1,4>{sfx}", **kw) == 44      # 24 keys at one CTA home
        _check_c(orc, eng, cols, s_, m_, aggs, [col(2)], f"{kname}<1,4>{sfx}", **kw)                   # a shared guess entry
        assert _check_c(orc, eng, cols, s_, m_, aggs, [col(2), "s3"], f"{kname}<2,4>{sfx}", **kw) == 20   # 7-byte keys
        _check_c(orc, eng, cols, s_, m_, aggs, ["s3", col(2)], f"{kname}<2,4>{sfx}", **kw)
    monkeypatch.setenv("IMM3_AGG_SLOTS", str(R.SMALL_SLOTS))
    for s_, m_ in ((NoSelect, every), (sel, mask)):
        assert _check_c(orc, eng, cols, s_, m_, aggs, [col(3)], f"{kname}<1,4>{sfx}", **kw) == 64       # the table exactly full
        with pytest.raises(Imm3Error) as e:
            eng.execute(Query("adv", s_, ProjectAgg(aggs, [col(4)])), **kw)                             # one group more
        assert e.value.status == L.ERR_UNSUPPORTED and "groups" in e.value.message, e.value.message
        assert _check_c(orc, eng, cols, s_, m_, aggs, [col(3)], f"{kname}<1,4>{sfx}", **kw) == 64       # the handle answers afterwards
        _check_c(orc, eng, cols, s_, m_, aggs, [col(1)], f"{kname}<1,4>{sfx}", **kw)
    monkeypatch.delenv("IMM3_AGG_SLOTS")
    assert _check_c(orc, eng, cols, NoSelect, every, aggs, [col(4)], f"{kname}<1,4>{sfx}", **kw) == 65


# ---- D. merge order across ranks ------------------------------------------------------------------------------------------

D_BLOCK, D_SEG, D_NSEG = 256, 8, 10                                        # 10 segments: canonical order = write order
D_PER = D_BLOCK * D_SEG + 1


def _merge_table(data):
    """g (and its PFOR_INT twin gp), per canonical segment s: 30 background keys throughout; X (8 keys) as the LAST rows of
    segment 0 in reverse order, absent from segments 1-2, the first rows of segments 3-9 in order and scattered after;
    Y (8 keys) only in segments 5-9; Z (4 keys) only as the last rows of segment 9."""
    rng = np.random.default_rng(31)
    n = D_NSEG * D_PER
    base = rng.choice(np.arange(1000, 100000, 7), 30, replace=False).astype(np.int32)
    X = np.arange(-8, 0, dtype=np.int32) * 1000
    Y = np.arange(1, 9, dtype=np.int32) * 7_000_000
    Z = np.array([I32_MIN, I32_MAX, 0, 5], np.int32)
    g = base[rng.integers(0, len(base), n)]
    for s in range(D_NSEG):
        a = s * D_PER
        seg = g[a:a + D_PER]
        if s == 0:
            seg[-len(X):] = X[::-1]
        if s >= 3:
            seg[:len(X)] = X
            pick = rng.random(D_PER) < 0.1
            pick[:len(X)] = False
            seg[pick] = X[rng.integers(0, len(X), int(pick.sum()))]
        if s >= 5:
            pick = rng.random(D_PER) < 0.1
            pick[:len(X)] = False
            seg[pick] = Y[rng.integers(0, len(Y), int(pick.sum()))]
        if s == D_NSEG - 1:
            seg[-len(Z):] = Z
    cols = {"g": g, "gp": g, "v": rng.integers(I32_MIN, I32_MAX, n, dtype=np.int64, endpoint=True).astype(np.int32),
            "b": rng.integers(-128, 128, n, dtype=np.int64).astype(np.int8)}
    write_table(data, "m", cols, ["g:DENSE_INT", "gp:PFOR_INT", "v:DENSE_INT", "b:DENSE_TINYINT"], D_BLOCK, D_SEG)
    return cols, X, Y


def _merge_cases():
    sel = Select("b", GT(-60))
    return [(sel_, [Count("v"), Min("v"), Max("v")], gb) for sel_ in (NoSelect, sel) for gb in (["g"], ["gp"], ["g", "b"])]


def _merge_worker(rank, world, data_dir, port, out_dir, mode):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch
    import torch.distributed as dist

    import oracle_lib as O
    from test_gpu_agg_global import _oracle, _same
    from immutable3_b200 import Engine, ProjectAgg, Query, SegmentManager
    from immutable3_b200.dist import CudaExecutor, ShardedEngine

    ndev = torch.cuda.device_count()
    dev = rank % ndev
    backend = "nccl" if (mode == "device" and ndev >= world) else "gloo"
    if backend == "nccl":
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    os.environ["IMM3_COMM_TIMEOUT_MS"] = "10000"
    try:
        with SegmentManager(data_dir, device=dev, rank=rank, world=world) as sm, O.Oracle(data_dir) as whole:
            if mode == "device":
                sm.comm_connect()
            eng = Engine(sm)
            sh = ShardedEngine(CudaExecutor(eng), collective_device="cuda" if backend == "nccl" else "cpu")
            for sel, aggs, gb in _merge_cases():
                q = Query("m", sel, ProjectAgg(aggs, gb))
                exp = _oracle(whole, "m", sel, aggs, gb)
                res = sh.execute_agg(q)
                _same(res.columns, exp, (mode, rank, sel, aggs, gb))
                if mode == "device":
                    with eng.execute_agg_global(q) as r:
                        _same(r.columns(), exp, (rank, sel, aggs, gb))
                        assert r.route.endswith("agg_exchange;agg_init;agg_merge;agg_compact"), r.route
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world, mode", [(2, "device"), (3, "device"), (2, "host"), (3, "host")])
def test_merge_order_across_ranks(tmp_path, world, mode):
    from immutable3_b200.dist import shard_range

    data = tmp_path / "data"
    cols, X, Y = _merge_table(data)
    g = cols["g"]
    # premise: the ranks' first-appearance orders disagree - Y is absent from rank 0, X is first on rank 1 in the order
    # opposite to rank 0's, where X only appears late
    order = lambda a: list(dict.fromkeys(a.tolist()))
    slices = [g[b * D_PER:e * D_PER] for b, e in (shard_range(D_NSEG, r, world) for r in range(world))]
    o0, o1 = order(slices[0]), order(slices[1])
    assert not set(Y.tolist()) & set(o0)
    assert [k for k in o0 if k in set(X.tolist())] == X[::-1].tolist() and [k for k in o1 if k in set(X.tolist())] == X.tolist()
    assert o0.index(int(X[-1])) >= len(o0) - len(X) and o1[:len(X)] == X.tolist()
    port = 51700 + (os.getpid() % 2000) + world + (10 if mode == "host" else 0)
    mp.spawn(_merge_worker, args=(world, str(data), port, str(tmp_path), mode), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))
