"""Real OR's select-tree expansion and its independent reference, without a GPU.

select_dnf turns the select tree into the conjunctions imm3_query_begin_dnf runs; select_tree_ref.eval_tree walks the tree
itself.  On random trees the two must agree row for row: eval_tree's mask equals the union of the oracle's selection
bitmaps (orc_filter_bitmap) over select_dnf's conjunctions.  A wrong expansion, or a wrong reference, fails here before any
GPU test trusts either.  Also pinned: what a tree that expands to more than MAX_OR_TERMS conjunctions does."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
from helpers import STATES, conj, make_table, oracle_preds
from immutable3_b200 import (EQ, GT, LT, OPEN_HOST_ONLY, And, Engine, Imm3Error, Match, NoSelect, Or, Project, Query, SegmentManager,
                             Select, select_dnf)
from immutable3_b200 import _lib as L
from immutable3_b200.engine import MAX_OR_TERMS
from select_tree_ref import can_hold, canonical_columns, dnf_size, eval_tree, random_tree

NAMES = np.array([b"alice", b"bobby", b"carol", b"dave_", b"erin#"], "S5")
COLS = ["id", "state", "age", "name"]


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    d = tmp_path_factory.mktemp("or_tree_host")
    rng = np.random.default_rng(5)
    n = 12_345
    # 25 segments of 501 rows: canonical (file-name) order is not write order
    make_table(d, "t", n, 50, 10, seed=3, extra_cols=[("name:DENSE_STRING:size=5", NAMES[rng.integers(0, 5, n)])])
    with O.Oracle(d) as orc:
        yield d, orc, canonical_columns(orc, "t", COLS)


def union_of_bitmaps(orc, table, select):
    n = orc.nrows(table)
    keep = np.zeros(n, bool)
    for term in select_dnf(select):
        words, _ = orc.filter_bitmap(table, oracle_preds(conj(*term)))
        keep |= np.unpackbits(words.view(np.uint8), bitorder="little")[:n].astype(bool)
    return keep


def leaf_of(cols):
    ids = cols["id"]

    def leaf(rng):
        k = rng.integers(0, 9)
        if k == 0:
            return Select("age", GT(float(rng.integers(-140, 140))))
        if k == 1:
            return Select("age", LT(float(rng.integers(-140, 140)) + 0.5))
        if k == 2:
            return Select("age", EQ(float(rng.integers(-130, 130))))
        if k in (3, 4):
            q = float(np.quantile(ids, rng.random()))
            return Select("id", GT(q)) if k == 3 else Select("id", LT(q))
        if k == 5:
            return Select("state", Match([str(s) for s in rng.choice(STATES, size=int(rng.integers(1, 8)))] + (["CAL"] if rng.random() < 0.2 else [])))
        if k == 6:
            return Select("name", Match([v.decode() for v in rng.choice(NAMES, size=int(rng.integers(1, 3)))] + (["bob"] if rng.random() < 0.3 else [])))
        if k == 7:
            return Select("name", Match(["al", "alice_"]))                                 # wrong lengths: never holds
        return NoSelect if rng.random() < 0.3 else Select("age", GT(-129))                  # (-129 narrows to 127: never holds)

    return leaf


def test_random_trees_agree_with_the_union_of_their_conjunctions(world):
    d, orc, cols = world
    rng = np.random.default_rng(2718)
    leaf = leaf_of(cols)
    sizes = set()
    for _ in range(300):
        tree = random_tree(rng, leaf)
        terms = select_dnf(tree)
        assert len(terms) == dnf_size(tree) <= MAX_OR_TERMS
        sizes.add(len(terms))
        mask = eval_tree(cols, tree)
        keep = union_of_bitmaps(orc, "t", tree)
        if not np.array_equal(mask, keep):
            bad = int(np.flatnonzero(mask != keep)[0])
            raise AssertionError(f"{tree}: row {bad} tree {mask[bad]} conjunctions {keep[bad]}")
    assert max(sizes) >= 8 and 1 in sizes, sorted(sizes)


def test_fixed_trees(world):
    """Shapes whose meaning is easy to state, with the row count numpy gives directly."""
    d, orc, cols = world
    age, st, ids = cols["age"].astype(np.int64), cols["state"], cols["id"].astype(np.int64)
    a, b, c = Select("age", LT(10)), Select("state", Match(["CA", "TX"])), Select("id", GT(20_000))
    cases = [(Or(a, b), (age < 10) | np.isin(st, [b"CA", b"TX"])),
             (And(Or(a, b), c), ((age < 10) | np.isin(st, [b"CA", b"TX"])) & (ids > 20_000)),
             (And(c, Or(a, NoSelect)), ids > 20_000),
             (Or(a, a), age < 10),
             (Or(Select("age", GT(-129)), a), age < 10),                                       # a term narrowed away
             (Or(Select("state", Match(["C"])), Select("state", Match(["CAX"]))), np.zeros(len(age), bool))]
    for tree, want in cases:
        assert np.array_equal(eval_tree(cols, tree), want), tree
        assert np.array_equal(union_of_bitmaps(orc, "t", tree), want), tree


def test_can_hold_is_the_planners_narrowing(world):
    d, orc, cols = world
    assert can_hold([Select("age", GT(10)), Select("age", LT(12))], cols)
    assert not can_hold([Select("age", GT(10)), Select("age", LT(11))], cols)
    assert not can_hold([Select("age", GT(-129))], cols)                                     # age > 127
    assert can_hold([Select("age", GT(-128.5))], cols)                                       # age > -128
    assert not can_hold([Select("state", Match(["CA"])), Select("state", Match(["TX"]))], cols)
    assert not can_hold([Select("name", Match(["bob"]))], cols)
    assert can_hold([Select("id", LT(-5))], cols)                                            # no row, but a range
    assert can_hold([], cols)


def sixteen(k=0):
    """And of four Ors: 16 conjunctions; with k > 0 one more Or level on the last operand."""
    p = [Select("age", GT(i)) for i in range(8 + k)]
    last = Or(p[6], p[7]) if k == 0 else Or(p[6], Or(p[7], p[8]))
    return And(Or(p[0], p[1]), And(Or(p[2], p[3]), And(Or(p[4], p[5]), last)))


def test_more_than_max_or_terms(world):
    """In Python a tree of more than MAX_OR_TERMS (16) conjunctions raises Imm3Error(ERR_UNSUPPORTED) in select_dnf, before
    any call; the C entry point given 17 terms returns IMM3_ERR_INVALID_ARG.  16 pass both."""
    d, orc, cols = world
    assert len(select_dnf(sixteen())) == MAX_OR_TERMS == 16
    with pytest.raises(Imm3Error) as e:
        select_dnf(sixteen(1))
    assert e.value.status == L.ERR_UNSUPPORTED and "24 conjunctions" in str(e.value)
    with SegmentManager(d, flags=OPEN_HOST_ONLY) as sm:
        eng = Engine(sm)
        with pytest.raises(Imm3Error) as e:
            eng.execute(Query("t", sixteen(1), Project(["id"])), real_or=True)
        assert e.value.status == L.ERR_UNSUPPORTED
        with pytest.raises(Imm3Error) as e:                                                   # 16 reach the library (no device here)
            eng.execute(Query("t", sixteen(), Project(["id"])), real_or=True)
        assert e.value.status == L.ERR_STATE
        lib = L.lib()
        for nterms, want in ((17, L.ERR_INVALID_ARG), (16, L.ERR_STATE)):
            preds = (L.Pred * nterms)()
            for i in range(nterms):
                preds[i].col, preds[i].op, preds[i].num = b"age", L.OP_GT, float(i)
            sizes = (C.c_int32 * nterms)(*([1] * nterms))
            proj = L.cstr_array(["id"])
            out = C.c_void_p()
            st = lib.imm3_query_begin_dnf(sm.handle, b"t", preds, sizes, nterms, C.cast(proj, C.POINTER(C.c_char_p)), 1, 0, C.byref(out))
            assert st == want, (nterms, st, lib.imm3_last_error())
