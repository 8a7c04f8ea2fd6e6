"""Validation of aggregates under predicates on sorted-int-codec (PFOR_INT) columns (imm3_query_agg_ext with
IMM3_AGG_ENCODED_FILTER), on a host-only handle: with the flag the queries pass validation and stop at the device
(IMM3_ERR_STATE: no CPU fallback); without it, and on the parity entry points, they keep today's refusal; tables with blocks
of more than 1024 rows are refused before any device work; Python's `encoded_filter` and `sum_avg` stay independent."""
import ctypes as C

import numpy as np
import pytest

from helpers import conj, make_table
from immutable3_b200 import (Avg, Count, EQ, Engine, GT, Imm3Error, LT, Match, Max, Min, NoSelect, OPEN_HOST_ONLY, ProjectAgg, Query,
                             SegmentManager, Select, Sum)
from immutable3_b200 import _lib as L


@pytest.fixture(scope="module")
def sm(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg_enc_filter_host")
    n = 3000
    make_table(d, "p", n, 128, 3, seed=4, id_codec="PFOR_INT", id_mode="steps",
               extra_cols=[("e0:PFOR_INT", np.arange(n, dtype=np.int32) * 3)])
    make_table(d, "t", n, 64, 5, seed=2)                                                   # dense id
    make_table(d, "big", n, 2048, 1, seed=4, id_codec="PFOR_INT", id_mode="steps")       # blocks of 2048 rows
    s = SegmentManager(d, flags=OPEN_HOST_ONLY)
    yield s
    s.close()


def _status(sm, table, sel, aggs, group_by, **kw):
    with pytest.raises(Imm3Error) as e:
        Engine(sm).execute(Query(table, sel, ProjectAgg(aggs, group_by)), **kw)
    return e.value.status, e.value.message


WINDOW = conj(Select("id", GT(100)), Select("id", LT(2000)))
SELS = [WINDOW,
        Select("id", GT(5)),
        Select("id", LT(5)),
        Select("id", EQ(0)),
        conj(WINDOW, Select("age", GT(18))),                                               # mixed with a dense predicate
        conj(WINDOW, Select("state", Match(["CA"]))),
        conj(Select("id", GT(10)), Select("e0", LT(4000)))]                                # two encoded columns
SHAPES = [([Count("id"), Min("age"), Max("age")], ["state"]),
          ([Min("id"), Max("id")], []),                                                    # the filtered column aggregated
          ([Count("age")], ["id"]),                                                        # ... and grouped
          ([Min("age"), Max("e0"), Count("id")], ["state", "age"])]


@pytest.mark.parametrize("sel", SELS)
@pytest.mark.parametrize("aggs, group_by", SHAPES)
def test_flag_passes_validation_and_parity_refuses(sm, sel, aggs, group_by):
    assert _status(sm, "p", sel, aggs, group_by, encoded_filter=True)[0] == L.ERR_STATE
    assert _status(sm, "p", sel, aggs, group_by, encoded_filter=True, sum_avg=True)[0] == L.ERR_STATE
    old = _status(sm, "p", sel, aggs, group_by)
    assert old[0] == L.ERR_UNSUPPORTED and "predicate on a sorted-int-codec column" in old[1]
    assert _status(sm, "p", sel, aggs, group_by, sum_avg=True) == old                     # _ext without the bit: word for word


def test_entry_points_and_flag_bits(sm):
    lib = L.lib()
    arr = (L.Agg * 1)()
    arr[0].col, arr[0].op = b"age", L.AGG_MIN
    preds = (L.Pred * 1)()
    preds[0].col, preds[0].op, preds[0].num = b"id", L.OP_GT, 5.0
    groups = L.cstr_array([])
    g = C.cast(groups, C.POINTER(C.c_char_p))
    out = C.c_void_p()

    def call(fn, *flags):
        return fn(sm.handle, b"p", preds, 1, arr, 1, g, 0, *flags, C.byref(out))

    msgs = []
    for fn, flags in ((lib.imm3_query_agg, ()), (lib.imm3_query_agg_global, ()), (lib.imm3_query_agg_ext, (0,)),
                      (lib.imm3_query_agg_ext, (L.AGG_FLAG_GLOBAL,))):
        assert call(fn, *flags) == L.ERR_UNSUPPORTED
        msgs.append(lib.imm3_last_error())
    assert len(set(msgs)) == 1 and b"not supported yet" in msgs[0]
    for flags in (L.AGG_FLAG_ENCODED_FILTER, L.AGG_FLAG_ENCODED_FILTER | L.AGG_FLAG_GLOBAL):
        assert call(lib.imm3_query_agg_ext, flags) == L.ERR_STATE
    for flags in (0x2, 0x8, 0x6, 0x80000004):
        assert call(lib.imm3_query_agg_ext, flags) == L.ERR_INVALID_ARG and b"flag" in lib.imm3_last_error()


def test_no_encoded_predicate_is_unaffected(sm):
    for table, sel in (("p", NoSelect), ("p", Select("age", GT(18))), ("t", Select("id", GT(5))), ("t", NoSelect)):
        for aggs, gb in (([Count("id"), Min("age")], ["state"]), ([Max("id")], [])):
            assert _status(sm, table, sel, aggs, gb, encoded_filter=True) == _status(sm, table, sel, aggs, gb)
    for kw in ({}, {"encoded_filter": True}):                                              # a refusal is the same refusal
        st, msg = _status(sm, "p", NoSelect, [Count("age")], ["id", "id"], **kw)
        assert st == L.ERR_UNSUPPORTED and "7 bytes" in msg


def test_blocks_over_1024_rows(sm):
    for aggs in ([Count("age")], [Min("id")]):
        st, msg = _status(sm, "big", Select("id", GT(5)), aggs, ["state"], encoded_filter=True)
        assert st == L.ERR_UNSUPPORTED and "1024" in msg
        st, msg = _status(sm, "big", Select("id", GT(5)), aggs, ["state"], encoded_filter=True, sum_avg=True)
        assert st == L.ERR_UNSUPPORTED and "1024" in msg
    # without an encoded predicate the flag changes nothing: a Count reads no encoded column and takes the dense path
    assert _status(sm, "big", Select("age", GT(5)), [Count("age")], ["state"], encoded_filter=True)[0] == L.ERR_STATE


def test_encoded_filter_and_sum_avg_are_independent(sm):
    for aggs in ([Sum("age")], [Avg("id"), Count("id")]):
        for sel in (WINDOW, NoSelect):
            st, msg = _status(sm, "p", sel, aggs, ["state"], encoded_filter=True)
            assert (st, msg) == _status(sm, "t", NoSelect, aggs, ["state"])                # the parity path's refusal
            assert st == L.ERR_UNSUPPORTED and "Unknown Aggregate type" in msg
        assert _status(sm, "p", WINDOW, aggs, ["state"], encoded_filter=True, sum_avg=True)[0] == L.ERR_STATE
        st, msg = _status(sm, "p", WINDOW, aggs, ["state"], sum_avg=True)
        assert st == L.ERR_UNSUPPORTED and "predicate" in msg
    eng = Engine(sm)
    q = Query("p", WINDOW, ProjectAgg([Min("age")], []))
    for call in (lambda: eng.begin(q, encoded_filter=True), lambda: eng.execute_agg_global(q, encoded_filter=True)):
        with pytest.raises(Imm3Error) as e:
            call()
        assert e.value.status == L.ERR_STATE
