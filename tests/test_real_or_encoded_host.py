"""Validation of real OR over sorted-int-codec (PFOR_INT) columns (imm3_query_begin_dnf_ext with IMM3_DNF_ENCODED_FILTER), on a
host-only handle: unknown flag bits are refused; flags = 0 is imm3_query_begin_dnf word for word; the term limits hold; tables
with blocks of more than 1024 rows are refused before any device work; everything else passes validation and stops at the
device (IMM3_ERR_STATE: no CPU fallback); Python's `encoded_filter` reaches the new symbol only with `real_or`."""
import ctypes as C

import numpy as np
import pytest

from helpers import conj, make_table
from immutable3_b200 import Engine, GT, Imm3Error, LT, Match, OPEN_HOST_ONLY, Or, Project, Query, SegmentManager, Select
from immutable3_b200 import _lib as L


@pytest.fixture(scope="module")
def sm(tmp_path_factory):
    d = tmp_path_factory.mktemp("real_or_enc_host")
    n = 3000
    make_table(d, "p", n, 128, 3, seed=4, id_codec="PFOR_INT", id_mode="steps",
               extra_cols=[("e0:PFOR_INT", np.arange(n, dtype=np.int32) * 3)])
    make_table(d, "big", n, 2048, 1, seed=4, id_codec="PFOR_INT", id_mode="steps")       # blocks of 2048 rows
    s = SegmentManager(d, flags=OPEN_HOST_ONLY)
    yield s
    s.close()


def _preds(terms):
    flat = [p for t in terms for p in t]
    arr = (L.Pred * max(1, len(flat)))()
    for i, (col, op, num) in enumerate(flat):
        arr[i].col, arr[i].op, arr[i].num = col, op, float(num)
    return arr, (C.c_int32 * max(1, len(terms)))(*[len(t) for t in terms])


def _call(sm, table, terms, flags=None, nterms=None, proj=(b"id",), sizes=None):
    """(status, message) of imm3_query_begin_dnf (flags None) or imm3_query_begin_dnf_ext."""
    lib = L.lib()
    preds, sz = _preds(terms)
    cols = L.cstr_array(list(proj))
    out = C.c_void_p()
    args = (sm.handle, table, preds, sizes if sizes is not None else sz, len(terms) if nterms is None else nterms,
            C.cast(cols, C.POINTER(C.c_char_p)), len(proj), 0)
    st = lib.imm3_query_begin_dnf(*args, C.byref(out)) if flags is None else lib.imm3_query_begin_dnf_ext(*args, flags, C.byref(out))
    return st, lib.imm3_last_error()


ID_WINDOW = [(b"id", L.OP_GT, 100), (b"id", L.OP_LT, 900)]
CASES = [("p", [ID_WINDOW, [(b"id", L.OP_GT, 2500)]]),                                      # two windows on the encoded id
         ("p", [[(b"id", L.OP_LT, 10)], [(b"age", L.OP_EQ, 3)]]),                            # encoded OR dense
         ("p", [ID_WINDOW + [(b"age", L.OP_GT, 50)], [(b"age", L.OP_LT, 2)]]),
         ("p", [[(b"id", L.OP_GT, 10)], [(b"e0", L.OP_LT, 400)], [(b"id", L.OP_EQ, 0)]]),    # two encoded columns
         ("p", [[(b"age", L.OP_GT, 90)], [(b"age", L.OP_LT, 5)]]),                           # dense only
         ("p", [[(b"id", L.OP_GT, 10), (b"id", L.OP_LT, 5)], [(b"age", L.OP_LT, 5)]]),       # a term that drops out
         ("p", [ID_WINDOW]),                                                                 # a single term
         ("p", [ID_WINDOW, [(b"nope", L.OP_GT, 1)]]),                                        # unknown column
         ("nope", [ID_WINDOW, [(b"age", L.OP_GT, 1)]]),                                      # unknown table
         ("big", [ID_WINDOW, [(b"age", L.OP_GT, 1)]])]


@pytest.mark.parametrize("ci", range(len(CASES)))
def test_flags_zero_is_the_dnf_entry_point(sm, ci):
    table, terms = CASES[ci]
    assert _call(sm, table.encode(), terms, flags=0) == _call(sm, table.encode(), terms)


def test_flag_passes_validation(sm):
    for table, terms in CASES[:7]:
        assert _call(sm, table.encode(), terms, flags=L.DNF_FLAG_ENCODED_FILTER)[0] == L.ERR_STATE, (table, terms)
    assert _call(sm, b"p", CASES[7][1], flags=L.DNF_FLAG_ENCODED_FILTER) == _call(sm, b"p", CASES[7][1])
    assert _call(sm, b"nope", CASES[8][1], flags=L.DNF_FLAG_ENCODED_FILTER) == _call(sm, b"nope", CASES[8][1])


def test_unknown_flag_bits(sm):
    for flags in (0x1, 0x2, 0x8, 0x6, 0x80000004):
        st, msg = _call(sm, b"p", CASES[0][1], flags=flags)
        assert st == L.ERR_INVALID_ARG and b"flag" in msg, (flags, st, msg)


def test_term_limits(sm):
    many = [[(b"id", L.OP_GT, i)] for i in range(17)]
    for flags in (0, L.DNF_FLAG_ENCODED_FILTER):
        st, msg = _call(sm, b"p", many, flags=flags)
        assert (st, msg) == _call(sm, b"p", many) and st == L.ERR_INVALID_ARG and b"16" in msg
        assert _call(sm, b"p", many[:16], flags=flags)[0] == L.ERR_STATE                   # 16 terms pass
        st, msg = _call(sm, b"p", CASES[0][1], flags=flags, nterms=0)
        assert st == L.ERR_INVALID_ARG
        st, msg = _call(sm, b"p", CASES[0][1], flags=flags, sizes=(C.c_int32 * 2)(2, -1))
        assert st == L.ERR_INVALID_ARG and b"term 1" in msg


def test_blocks_over_1024_rows(sm):
    for terms in (CASES[9][1], [[(b"id", L.OP_LT, 5)], [(b"id", L.OP_GT, 2900)]]):
        st, msg = _call(sm, b"big", terms, flags=L.DNF_FLAG_ENCODED_FILTER)
        assert st == L.ERR_UNSUPPORTED and b"1024" in msg, msg
    # a single term, or terms on dense columns only, are not the block-space disjunction: the flag changes nothing
    for terms in ([ID_WINDOW], [[(b"age", L.OP_GT, 90)], [(b"age", L.OP_LT, 5)]]):
        assert _call(sm, b"big", terms, flags=L.DNF_FLAG_ENCODED_FILTER) == _call(sm, b"big", terms)


def test_python_keywords(sm, monkeypatch):
    eng = Engine(sm)
    q = Query("p", Or(Select("id", LT(10)), Select("state", Match(["CA"]))), Project(["id"]))
    seen = []
    lib = L.lib()
    real_dnf, real_ext = lib.imm3_query_begin_dnf, lib.imm3_query_begin_dnf_ext

    class Spy:
        def __getattr__(self, name):
            return getattr(lib, name)

        def imm3_query_begin_dnf(self, *a):
            seen.append(("dnf", None))
            return real_dnf(*a)

        def imm3_query_begin_dnf_ext(self, *a):
            seen.append(("ext", a[-2]))
            return real_ext(*a)

    monkeypatch.setattr(eng, "_lib", Spy())
    for call in (lambda: eng.execute(q, real_or=True, encoded_filter=True), lambda: eng.begin(q, real_or=True, encoded_filter=True)):
        with pytest.raises(Imm3Error) as e:
            call()
        assert e.value.status == L.ERR_STATE
    assert seen == [("ext", L.DNF_FLAG_ENCODED_FILTER)] * 2
    seen.clear()
    with pytest.raises(Imm3Error):
        eng.execute(q, real_or=True)
    assert seen == [("dnf", None)]
    seen.clear()
    with pytest.raises(Imm3Error):                                                         # no real_or: encoded_filter is ignored
        eng.execute(Query("p", conj(Select("id", GT(5)), Select("id", LT(90))), Project(["id"])), encoded_filter=True)
    assert seen == []
