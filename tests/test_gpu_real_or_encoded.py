"""Real OR over sorted-int-codec (PFOR_INT) columns on the GPU (imm3_query_begin_dnf_ext with IMM3_DNF_ENCODED_FILTER): every
term runs the block filter front and blocks_or_merge_kernel ORs its per-block selection into the first term's.  Expected rows
are the oracle's unfiltered rows under the OR of its per-term selection bitmaps (test_gpu_real_or.expected), cut at LIMIT in
canonical order; also against the dense-id twin, numpy at 40 M rows, and across segment-sharded ranks."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

import oracle_lib as O
from helpers import conj, make_table, oracle_preds
from immutable3_b200 import And, EQ, Engine, GT, LT, Match, Or, Project, Query, SegmentManager, Select
from immutable3_b200 import _lib as L
from test_gpu_real_or import QUERIES, expected

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("real_or_enc")
    rng = np.random.default_rng(17)
    n = 70_001
    extra = [("name:DENSE_STRING:size=5", np.array([b"alice", b"bobby", b"carol", b"dave_", b"erin#"], "S5")[rng.integers(0, 5, n)]),
             ("score:DENSE_INT", rng.integers(-1000, 1000, n).astype(np.int32))]
    make_table(d, "t", n, 100, 7, seed=8, extra_cols=extra)                                   # test_gpu_real_or's tables
    make_table(d, "p", 40_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    make_table(d, "q", 30_000, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps",         # quad kernel
               extra_cols=[("e0:PFOR_INT", (np.arange(30_000) * 3 + 11).astype(np.int32))])
    make_table(d, "pl", 60_000, 1024, 14, seed=4, id_codec="PFOR_INT", id_mode="sorted")      # lane kernel
    make_table(d, "pk", 30_001, 1000, 3, seed=5, id_codec="PFOR_INT", id_mode="sorted")       # blocks of 1000 rows, a 1-row tail
    make_table(d, "p32", 5_001, 32, 40, seed=6, id_codec="PFOR_INT", id_mode="sorted")        # blocks of 32 rows, a 1-row tail
    make_table(d, "tp", 50_000, 1024, 7, seed=6, id_codec="PFOR_INT", id_mode="steps")        # twins: same rows, encoded / dense id
    make_table(d, "td", 50_000, 1024, 7, seed=6, id_codec="DENSE_INT", id_mode="steps")
    orc, sm = O.Oracle(d), SegmentManager(d)
    yield d, orc, sm
    sm.close()
    orc.close()


def run(orc, eng, table, sel, proj, limit=0, route=None, encoded=True):
    """The disjunction against the oracle (rows and order); returns the route."""
    exp = expected(orc, table, sel, proj, limit)
    with eng.execute(Query(table, sel, Project(proj, limit)), real_or=True, encoded_filter=encoded) as got:
        assert got.nrows == len(exp[0]), (table, sel, limit, got.nrows, len(exp[0]), got.route)
        for c in range(len(proj)):
            assert np.array_equal(got.column(c), exp[c]), (table, sel, proj[c], limit, got.route)
        r = got.route
        assert got.kernel_launches == (len(r.split(";")) if r else 0), (got.kernel_launches, r)
    if route is not None:
        assert route in r, (route, r)
    return r


def ids_of(orc, table):
    return np.asarray(orc.query(table, [], ["id"]).columns[0]).astype(np.int64)


def window(lo, hi):
    return conj(Select("id", GT(int(lo))), Select("id", LT(int(hi))))


def window_pairs(ids, block):
    n, lo, hi = len(ids), int(ids.min()), int(ids.max())
    at = lambda i: int(ids[min(max(i, 0), n - 1)])
    B = block
    return [(window(at(B + 5), at(B + 300)), window(at(3 * B + 10), at(5 * B - 1))),          # disjoint
            (window(at(B - 1), at(2 * B)), window(at(2 * B) - 1, at(3 * B))),                # adjacent, on block edges
            (window(at(31), at(32 * 5)), window(at(32 * 3), at(32 * 9) + 1)),                # overlapping, on mini-block edges
            (window(at(B // 2), at(4 * B + 7)), window(at(B + 40), at(2 * B + 33))),         # nested
            (window(at(n // 2), at(n // 2 + 700)), window(at(n // 2), at(n // 2 + 700))),  # the same term twice
            (window(at(n // 2), at(n // 2) + 1), window(at(100), at(900))),                # a term that can never hold drops out
            (window(lo - 1, hi + 1), window(at(100), at(200))),                              # a window covering the table
            (Select("id", EQ(lo)), Select("id", EQ(hi))),                                    # EQ on the extremes
            (Select("id", LT(at(n // 4))), Select("id", GT(at(3 * n // 4))))]


@pytest.mark.parametrize("table, block", [("p", 1024), ("q", 1024), ("pl", 1024), ("pk", 1000), ("p32", 32)])
def test_two_windows(world, table, block):
    d, orc, sm = world
    eng = Engine(sm)
    ids = ids_of(orc, table)
    for i, (a, b) in enumerate(window_pairs(ids, block)):
        for proj in (["id"], ["id", "age"]):
            r = run(orc, eng, table, Or(a, b), proj)
            assert ("blocks_or_merge" in r) == (i != 5), r                                    # (5: one term remains)
        run(orc, eng, table, Or(a, b), ["id", "state"], limit=77)
    # three and four windows
    at = lambda i: int(ids[min(i, len(ids) - 1)])
    wins = [window(at(i * len(ids) // 4 + 3), at(i * len(ids) // 4 + 500)) for i in range(4)]
    r = run(orc, eng, table, Or(wins[0], Or(wins[1], Or(wins[2], wins[3]))), ["id"])
    assert r.count("blocks_or_merge") == 3, r


def test_encoded_and_dense_terms(world):
    d, orc, sm = world
    eng = Engine(sm)
    ids = ids_of(orc, "q")
    w = window(ids[2000], ids[9000])
    run(orc, eng, "q", Or(w, Select("age", GT(90))), ["id", "age"], route="blocks_or_merge")
    run(orc, eng, "q", Or(And(w, Select("age", GT(50))), Select("state", Match(["CA"]))), ["id", "state"], route="blocks_or_merge")
    run(orc, eng, "q", Or(Select("state", Match(["CA"])), w), ["id"], route="blocks_or_merge")       # the dense term carries the emit
    run(orc, eng, "q", Or(window(ids[100], ids[5000]), Select("e0", LT(3 * 20_000))), ["id", "e0"], route="blocks_or_merge")
    run(orc, eng, "q", Or(conj(w, Select("e0", GT(3 * 5000))), Select("e0", LT(40))), ["e0"], route="blocks_or_merge")


def _block_counts(ids, lo, hi, block):
    m = (ids > lo) & (ids < hi)
    pad = (-len(m)) % block
    return np.concatenate([m, np.zeros(pad, bool)]).reshape(-1, block).sum(1)


def test_merge_branches(world):
    """Two windows whose per-block selections meet each branch of the merge, asserted from the ids."""
    d, orc, sm = world
    eng = Engine(sm)
    ids = ids_of(orc, "pl")
    B = 1024
    v = lambda b, r: int(ids[b * B + r])
    nb = (len(ids) + B - 1) // B
    full = np.array([min(B, len(ids) - b * B) for b in range(nb)])
    cases = [((v(5, 100), v(5, 300)), (v(5, 600), v(5, 800)), 5, "pp_partial"),
             ((v(7, 0) - 1, v(7, 600)), (v(7, 500), v(8, 0)), 7, "pp_full"),
             ((v(20, 0), v(20, 10)), (v(9, 100), v(9, 900)), 9, "empty_partial"),
             ((v(11, 0) - 1, v(12, 0)), (v(11, 100), v(11, 900)), 11, "full_partial"),
             ((v(13, 0) - 1, v(14, 0)), (v(13, 0) - 1, v(14, 0)), 13, "full_full"),
             ((v(15, 200), v(15, 700)), (v(30, 0), v(31, 0)), 15, "partial_empty")]
    for (a, b, blk, kind) in cases:
        ca, cb = _block_counts(ids, *a, B)[blk], _block_counts(ids, *b, B)[blk]
        union = int((((ids > a[0]) & (ids < a[1])) | ((ids > b[0]) & (ids < b[1])))[blk * B:(blk + 1) * B].sum())
        want = {"pp_partial": 0 < ca < B and 0 < cb < B and union < B, "pp_full": 0 < ca < B and 0 < cb < B and union == full[blk],
                "empty_partial": ca == 0 and 0 < cb < B, "full_partial": ca == full[blk] and 0 < cb < B,
                "full_full": ca == cb == full[blk], "partial_empty": 0 < ca < B and cb == 0}[kind]
        assert want, (kind, ca, cb, union)
        for proj in (["id"], ["id", "age"]):
            run(orc, eng, "pl", Or(window(*a), window(*b)), proj, route="blocks_or_merge")


@pytest.mark.parametrize("prune", [True, False])
def test_stale_words_are_never_read(world, monkeypatch, prune):
    """Disjunctions whose edges cut blocks X and Y write their words; C4 Project queries write other blocks' words; then
    disjunctions that select X and Y wholly or not at all must not see any of them."""
    d, orc, sm = world
    eng = Engine(sm)
    if not prune:
        monkeypatch.setenv("IMM3_NO_PRUNE", "1")
    ids = ids_of(orc, "pl")
    X, Y = 5, 17
    mid = lambda b: int(ids[b * 1024 + 500])
    lo_, hi_ = lambda b: int(ids[b * 1024]), lambda b: int(ids[b * 1024 + 1023])
    cut = Or(window(mid(X), mid(X) + 300), window(mid(Y) - 300, mid(Y)))
    wholly = [Or(window(lo_(X) - 1, hi_(X) + 1), window(lo_(Y) - 1, hi_(Y) + 1)),             # X and Y wholly selected
              Or(window(hi_(X), lo_(X + 1) + 3), window(hi_(Y), lo_(Y + 1) + 3)),              # not at all
              Or(window(lo_(X) - 1, hi_(X) + 1), window(hi_(Y), lo_(Y + 1) + 3))]              # X wholly, Y not at all
    for rnd in range(3):
        run(orc, eng, "pl", cut, ["id"])
        for k in range(3):
            lo, hi = mid(2 + 7 * k + rnd), mid(9 + 7 * k + rnd)
            exp = orc.query("pl", oracle_preds(window(lo, hi)), ["id"], limit=0)
            with eng.execute(Query("pl", window(lo, hi), Project(["id"]))) as r:
                assert r.nrows == exp.nrows and np.array_equal(r.column(0), exp.columns[0])
        for sel in wholly:
            run(orc, eng, "pl", sel, ["id"])
            run(orc, eng, "pl", sel, ["id", "age"])


ROUTE_CASES = [({}, "pl", "blocks_filter_lane/w="),
               ({"IMM3_NO_LANE": "1"}, "pl", "blocks_filter_quad/s="),
               ({"IMM3_NO_QUAD": "1"}, "pl", "blocks_filter/s="),
               ({"IMM3_LANE_WARPS": "4"}, "pl", "blocks_filter_lane/w=4/"),
               ({"IMM3_NO_PRUNE": "1"}, "pl", "blocks_filter_lane/w=")]


@pytest.mark.parametrize("ci", range(len(ROUTE_CASES)))
def test_filter_kernels(world, monkeypatch, ci):
    d, orc, sm = world
    env, table, kern = ROUTE_CASES[ci]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    eng = Engine(sm)
    ids = ids_of(orc, table)
    sel = Or(window(ids[3000], ids[9000]), window(ids[30_500], ids[41_000]))
    for proj in (["id"], ["id", "age"]):
        r = run(orc, eng, table, sel, proj)
        parts = r.split(";")
        assert sum(p.startswith(kern) for p in parts) == 2, r
        assert (parts.count("blocks_prune") == 2) == ("IMM3_NO_PRUNE" not in env), r
        assert parts[4 if "IMM3_NO_PRUNE" not in env else 2] == "blocks_or_merge", r


def test_without_block_statistics(world):
    d, orc, _ = world
    with SegmentManager(d, flags=L.OPEN_NO_STATS) as sm:
        eng = Engine(sm)
        ids = ids_of(orc, "pl")
        r = run(orc, eng, "pl", Or(window(ids[3000], ids[9000]), window(ids[30_500], ids[41_000])), ["id"])
        assert "blocks_prune" not in r and r.count("blocks_filter_lane") == 2 and "blocks_or_merge" in r, r


def test_both_emits(world, monkeypatch):
    d, orc, sm = world
    eng = Engine(sm)
    ids = ids_of(orc, "pl")
    sel = Or(window(ids[3000], ids[9000]), window(ids[30_500], ids[41_000]))
    assert run(orc, eng, "pl", sel, ["id"]).endswith("blocks_or_merge;blocks_scan_emit")
    assert run(orc, eng, "pl", sel, ["id", "age"]).endswith("blocks_or_merge;offset_scan;blocks_emit(blocks)")
    monkeypatch.setenv("IMM3_NO_SCANEMIT", "1")
    assert run(orc, eng, "pl", sel, ["id"]).endswith("blocks_or_merge;offset_scan;blocks_emit(blocks)")


@pytest.mark.parametrize("prefix", ["small", "off"])
def test_limits(world, monkeypatch, prefix):
    d, orc, sm = world
    if prefix == "small":
        monkeypatch.setenv("IMM3_PREFIX_ROWS", "4096")
    else:
        monkeypatch.setenv("IMM3_NO_PREFIX", "1")
    eng = Engine(sm)
    ids = ids_of(orc, "pl")
    sels = [Or(window(ids[3000], ids[9000]), window(ids[30_500], ids[41_000])),            # every term pruned: no prefix phase
            Or(window(ids[20_000], ids[20_900]), Select("age", LT(3))),                     # a dense term: a prefix phase
            Or(And(Select("state", Match(["CA"])), Select("age", EQ(7))), window(ids[50_000], ids[58_000]))]  # rows come late
    for k, sel in enumerate(sels):
        total = len(expected(orc, "pl", sel, ["id"], 0)[0])
        for limit in (0, 1, 77, total // 3, total, total + 1):
            r = run(orc, eng, "pl", sel, ["id", "age"], limit=limit)
            if prefix == "off" or k == 0:
                assert "/prefix" not in r, r
            elif limit in (1, 77):
                assert "blocks_or_merge/prefix" in r, r


@pytest.mark.parametrize("qi", range(len(QUERIES)))
def test_flag_changes_no_dense_disjunction(world, qi):
    d, orc, sm = world
    table, sel, proj = QUERIES[qi]
    eng = Engine(sm)
    for limit in (0, 1, 77, 10_000):
        q = Query(table, sel, Project(proj, limit))
        eng.execute(q, real_or=True).close()  # (the dense emit kernels learn the result's density per query shape: same history)
        with eng.execute(q, real_or=True) as a, eng.execute(q, real_or=True, encoded_filter=True) as b:
            assert (a.route, a.kernel_launches, a.nrows) == (b.route, b.kernel_launches, b.nrows)
            for c in range(len(proj)):
                assert np.array_equal(a.column(c), b.column(c))


def test_single_term_is_the_conjunction(world):
    d, orc, sm = world
    eng = Engine(sm)
    ids = ids_of(orc, "pl")
    for sel in (window(ids[3000], ids[9000]), Or(window(ids[3000], ids[9000]), window(ids[5], ids[5] + 1))):
        for proj, limit in ((["id"], 0), (["id", "age"], 10)):
            q = Query("pl", sel, Project(proj, limit))
            flat = Query("pl", window(ids[3000], ids[9000]), Project(proj, limit))
            with eng.execute(q, real_or=True, encoded_filter=True) as a, eng.execute(flat) as b:
                assert (a.route, a.kernel_launches, a.nrows) == (b.route, b.kernel_launches, b.nrows)
                assert np.array_equal(a.column(0), b.column(0))


def test_twins_agree(world):
    d, orc, sm = world
    eng = Engine(sm)
    ids = ids_of(orc, "tp")
    assert np.array_equal(ids, ids_of(orc, "td"))
    sels = [Or(window(ids[1000], ids[4000]), window(ids[20_000], ids[31_000])),
            Or(And(window(ids[1000], ids[40_000]), Select("age", GT(50))), Select("state", Match(["CA"]))),
            Or(Select("id", EQ(int(ids[0]))), Or(window(ids[7000], ids[7100]), Select("age", LT(2))))]
    for sel in sels:
        for proj, limit in ((["id"], 0), (["id", "state", "age"], 0), (["id"], 500)):
            with eng.execute(Query("tp", sel, Project(proj, limit)), real_or=True, encoded_filter=True) as a, \
                    eng.execute(Query("td", sel, Project(proj, limit)), real_or=True) as b:
                assert "blocks_or_merge" in a.route and "blocks_or_merge" not in b.route
                assert a.nrows == b.nrows and a.nrows > 0
                for c in range(len(proj)):
                    assert a.column(c).tobytes() == b.column(c).tobytes()


def test_40m_rows_against_numpy(tmp_path):
    from immutable3_b200.loader import synth_write

    n = 40_000_000
    synth_write(str(tmp_path), "t", n, 1024, 1000, L.CODEC_PFOR_INT)
    with O.Oracle(tmp_path) as orc:
        raw = orc.query("t", [], ["id", "state", "age"])
    ids, states, ages = (np.asarray(c) for c in raw.columns)
    i64 = ids.astype(np.int64)
    srt = np.sort(i64)
    q = lambda f: int(srt[int(f * (n - 1))])
    sel = Or(window(q(0.10), q(0.105)), Or(And(window(q(0.5), q(0.6)), Select("age", GT(60))), window(q(0.9), q(0.95))))
    keep = ((i64 > q(0.10)) & (i64 < q(0.105))) | ((i64 > q(0.5)) & (i64 < q(0.6)) & (ages > 60)) | ((i64 > q(0.9)) & (i64 < q(0.95)))
    sel2 = Or(window(q(0.2), q(0.3)), Or(window(q(0.25), q(0.4)), Select("state", Match(["CA"]))))
    keep2 = ((i64 > q(0.2)) & (i64 < q(0.3))) | ((i64 > q(0.25)) & (i64 < q(0.4))) | (states == b"CA")
    with SegmentManager(tmp_path) as sm:
        eng = Engine(sm)
        for s, k in ((sel, keep), (sel2, keep2)):
            for limit in (0, 1_000_000):
                with eng.execute(Query("t", s, Project(["id", "age"], limit)), real_or=True, encoded_filter=True) as got:
                    want = ids[k][:limit] if limit else ids[k]
                    assert got.route.count("blocks_or_merge") == 2, got.route
                    assert got.nrows == len(want) and np.array_equal(got.column(0), want)
                    assert np.array_equal(got.column(1), ages[k][:limit] if limit else ages[k])


# ---- across ranks (device exchange) --------------------------------------------------------------------------------------

def _worker(rank, world, data_dir, port, out_dir):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch.distributed as dist

    import oracle_lib as O
    from immutable3_b200 import Engine, Project, Query, SegmentManager
    from test_gpu_real_or import expected

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    os.environ["IMM3_PREFIX_ROWS"] = "4096"
    os.environ["IMM3_COMM_TIMEOUT_MS"] = "10000"
    try:
        with SegmentManager(data_dir, device=0, rank=rank, world=world) as sm, O.Oracle(data_dir) as whole:
            sm.comm_connect()
            eng = Engine(sm)
            ids = np.asarray(whole.query("p", [], ["id"]).columns[0]).astype(np.int64)
            at = lambda f: int(ids[int(f * (len(ids) - 1))])
            sels = [Or(window(at(0.1), at(0.3)), window(at(0.6), at(0.65))),
                    Or(window(at(0.45), at(0.55)), Select("age", LT(4))),
                    Or(window(ids[0] - 10, ids[0] - 1), Select("state", Match(["CA"]))),
                    Or(window(ids[0] - 10, ids[0] - 1), window(ids[-1] + 1, ids[-1] + 9))]   # nothing anywhere
            for sel in sels:
                for proj in (["id"], ["id", "age"]):
                    full = expected(whole, "p", sel, proj, 0)
                    limits = [0, 1, 10, 5000]
                    with eng.begin(Query("p", sel, Project(proj, 0)), real_or=True, encoded_filter=True) as h:
                        c0 = h.rank_counts[0]
                    limits += [c for c in (c0 - 1, c0, c0 + 1) if c > 0]                     # cuts at the rank boundary
                    for limit in limits:
                        want = [c[:limit] for c in full] if limit else full
                        with eng.begin(Query("p", sel, Project(proj, limit)), real_or=True, encoded_filter=True) as h:
                            assert h.global_count == len(want[0]), (rank, sel, limit, h.global_count, len(want[0]))
                            assert "blocks_or_merge" in h.route or h.route.startswith("count_exchange"), h.route   # (empty slice)
                            h.fetch(h.take)
                            for c in range(len(proj)):
                                got = h.column(c)
                                assert np.array_equal(got, want[c][h.global_offset:h.global_offset + h.take]), (rank, sel, limit, proj[c])
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world, nrows", [(2, 30_000), (3, 30_000), (3, 2000)])          # (2000 rows: one segment, empty slices)
def test_sharded(tmp_path, world, nrows):
    data = tmp_path / "data"
    make_table(data, "p", nrows, 1024, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    port = 46700 + (os.getpid() % 2000) + world + (5 if nrows < 10_000 else 0)
    mp.spawn(_worker, args=(world, str(data), port, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))
