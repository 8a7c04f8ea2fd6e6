"""Sum / Avg through imm3_query_agg_ext on a host-only handle: the queries the SUM instantiations take pass validation and
stop at the device (IMM3_ERR_STATE: no CPU fallback), the parity entry points keep refusing them, and the shapes the
extension does not take are refused before any device work.  The host merge of sharded Sum / Avg partials
(`merge_partials`, `sum_avg_partials`, `finish_sum_avg`) on hand-made partials."""
import ctypes as C

import numpy as np
import pytest

from helpers import make_table
from immutable3_b200 import (Avg, Count, Engine, GT, Imm3Error, Max, Min, NoSelect, OPEN_HOST_ONLY, ProjectAgg, Query, SegmentManager, Select,
                             Sum)
from immutable3_b200 import _lib as L
from immutable3_b200.dist import finish_sum_avg, merge_partials, sum_avg_partials


@pytest.fixture(scope="module")
def sm(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg_sum_host")
    make_table(d, "t", 3000, 64, 5, seed=2)
    make_table(d, "p", 3000, 128, 3, seed=4, id_codec="PFOR_INT", id_mode="steps")
    s = SegmentManager(d, flags=OPEN_HOST_ONLY)
    yield s
    s.close()


def _status(sm, table, sel, aggs, group_by, **kw):
    with pytest.raises(Imm3Error) as e:
        Engine(sm).execute(Query(table, sel, ProjectAgg(aggs, group_by)), **kw)
    return e.value.status, e.value.message


SHAPES = [([Sum("age")], []),
          ([Avg("id")], ["state"]),
          ([Sum("id"), Avg("age"), Count("id")], ["state"]),
          ([Avg("age"), Min("id"), Max("age")], ["state", "age"]),
          ([Sum("id")] * 7 + [Count("age")], ["age", "state", "age"]),     # 8 visible, the COUNT among them
          ([Sum("id")] * 7, ["state"])]                                     # 7 visible + the hidden COUNT


@pytest.mark.parametrize("table", ["t", "p"])
@pytest.mark.parametrize("aggs, group_by", SHAPES)
def test_sum_avg_pass_validation(sm, table, aggs, group_by):
    for sel in (NoSelect, Select("age", GT(18))):
        assert _status(sm, table, sel, aggs, group_by, sum_avg=True)[0] == L.ERR_STATE
        st, msg = _status(sm, table, sel, aggs, group_by)                   # the parity path still refuses
        assert st == L.ERR_UNSUPPORTED and "Unknown Aggregate type" in msg


def test_refusals(sm):
    st, msg = _status(sm, "t", NoSelect, [Sum("state")], [], sum_avg=True)
    assert st == L.ERR_UNSUPPORTED and "STRING" in msg
    st, msg = _status(sm, "t", NoSelect, [Avg("state"), Count("id")], ["age"], sum_avg=True)
    assert st == L.ERR_UNSUPPORTED and "STRING" in msg
    st, msg = _status(sm, "t", NoSelect, [Min("id")] * 7 + [Avg("age")], ["state"], sum_avg=True)   # 8 visible + a hidden COUNT
    assert st == L.ERR_UNSUPPORTED and "COUNT" in msg
    st, msg = _status(sm, "p", Select("id", GT(5)), [Sum("age")], ["state"], sum_avg=True)          # predicate on the encoded column
    assert st == L.ERR_UNSUPPORTED and "predicate" in msg
    st, msg = _status(sm, "t", NoSelect, [Min("state")], [], sum_avg=True)                          # as imm3_query_agg refuses it
    assert (st, msg) == _status(sm, "t", NoSelect, [Min("state")], [])


def test_unknown_flag_bits(sm):
    lib = L.lib()
    arr = (L.Agg * 1)()
    arr[0].col, arr[0].op = b"age", L.AGG_SUM
    groups = L.cstr_array([])
    out = C.c_void_p()
    for flags in (0x2, 0x80000000, 0x3):
        rc = lib.imm3_query_agg_ext(sm.handle, b"t", None, 0, arr, 1, C.cast(groups, C.POINTER(C.c_char_p)), 0, flags, C.byref(out))
        assert rc == L.ERR_INVALID_ARG and b"flag" in lib.imm3_last_error()
    for flags in (0, L.AGG_FLAG_GLOBAL):   # a world == 1 handle: the global form is the local one
        assert lib.imm3_query_agg_ext(sm.handle, b"t", None, 0, arr, 1, C.cast(groups, C.POINTER(C.c_char_p)), 0, flags, C.byref(out)) == L.ERR_STATE


def test_host_merge_of_sum_avg_partials():
    aggs = [Avg("age"), Sum("id"), Min("id")]
    plan, count = sum_avg_partials(aggs)
    assert plan == [Sum("age"), Sum("id"), Min("id"), Count("age")] and count == 3
    assert sum_avg_partials([Count("x"), Avg("y")]) == ([Count("x"), Sum("y")], 0)
    i8, f8 = np.int64, np.float64
    big = 2**31 - 1
    # rank partials of the plan: group key, sum(age), sum(id), min(id), count
    r0 = [np.array([b"CA", b"NY"]), np.array([-300, 7], i8), np.array([big * 3, 5], i8), np.array([4.0, -2.0], f8), np.array([3, 1], i8)]
    r1 = [np.array([b"TX", b"CA"]), np.array([1, 3], i8), np.array([9, big * 4], i8), np.array([0.0, 1.0], f8), np.array([1, 4], i8)]
    r2 = []                                                   # an empty slice
    merged = merge_partials([r0, r2, r1], 1, plan)
    assert list(merged[0]) == [b"CA", b"NY", b"TX"]
    assert list(merged[1]) == [-297, 7, 1] and list(merged[2]) == [big * 7, 5, 9] and merged[2].dtype == i8
    assert list(merged[3]) == [1.0, -2.0, 0.0] and list(merged[4]) == [7, 1, 1]
    out = finish_sum_avg(merged, 1, aggs, count)
    assert len(out) == 4                                      # the carried COUNT is dropped
    assert out[1].dtype == f8 and out[1].tobytes() == (np.array([-297.0, 7.0, 1.0]) / np.array([7.0, 1.0, 1.0])).tobytes()
    assert list(out[2]) == [big * 7, 5, 9] and list(out[3]) == [1.0, -2.0, 0.0]
    assert finish_sum_avg([], 1, aggs, count) == []
    huge = [np.array([1], i8), np.array([5], i8), np.array([1 + 2**32], i8)]
    with pytest.raises(Imm3Error) as e:
        finish_sum_avg(huge, 1, [Avg("age")], 1)
    assert e.value.status == L.ERR_UNSUPPORTED
