"""Validation of count / min / max ... group by over sorted-int-codec (PFOR_INT) columns, on a host-only handle: the queries
the block aggregation kernel takes pass validation and stop at the device (IMM3_ERR_STATE: no CPU fallback); the shapes it
does not take are refused before any device work."""
import numpy as np
import pytest

from helpers import make_table
from immutable3_b200 import Count, Engine, GT, Imm3Error, Max, Min, NoSelect, OPEN_HOST_ONLY, ProjectAgg, Query, SegmentManager, Select
from immutable3_b200 import _lib as L


@pytest.fixture(scope="module")
def sm(tmp_path_factory):
    d = tmp_path_factory.mktemp("agg_enc_host")
    n = 3000
    seq = np.arange(n, dtype=np.int32)
    make_table(d, "p", n, 128, 3, seed=4, id_codec="PFOR_INT", id_mode="steps",
               extra_cols=[(f"e{i}:PFOR_INT", seq * (i + 1)) for i in range(4)])
    make_table(d, "big", n, 2048, 1, seed=4, id_codec="PFOR_INT", id_mode="steps")   # blocks of 2048 rows
    s = SegmentManager(d, flags=OPEN_HOST_ONLY)
    yield s
    s.close()


def _status(sm, table, sel, aggs, group_by):
    with pytest.raises(Imm3Error) as e:
        Engine(sm).execute(Query(table, sel, ProjectAgg(aggs, group_by)))
    return e.value.status, e.value.message


@pytest.mark.parametrize("aggs, group_by", [
    ([Min("id")], []),
    ([Max("id")], ["state"]),
    ([Count("id"), Min("id"), Max("id")], ["state"]),
    ([Count("age")], ["id"]),
    ([Max("age")], ["id", "state", "age"]),                      # 4 + 2 + 1 key bytes
    ([Min("id"), Max("e0")], ["e1"]),
    ([Min("id"), Min("e0"), Max("e1")], ["e2"]),                 # four distinct encoded columns
])
def test_encoded_aggregates_pass_validation(sm, aggs, group_by):
    for sel in (NoSelect, Select("age", GT(18))):
        assert _status(sm, "p", sel, aggs, group_by)[0] == L.ERR_STATE


def test_refusals_before_any_device_work(sm):
    st, msg = _status(sm, "p", NoSelect, [Count("age")], ["id", "id"])                    # 8 key bytes
    assert st == L.ERR_UNSUPPORTED and "7 bytes" in msg
    st, msg = _status(sm, "p", Select("id", GT(5)), [Min("id")], [])                      # predicate on the encoded column
    assert st == L.ERR_UNSUPPORTED and "predicate" in msg
    st, msg = _status(sm, "p", NoSelect, [Min("id"), Max("e0"), Min("e1"), Max("e2")], ["e3"])  # a fifth encoded column
    assert st == L.ERR_UNSUPPORTED and "at most 4" in msg
    st, msg = _status(sm, "big", NoSelect, [Min("id")], ["state"])                        # blocks of more than 1024 rows
    assert st == L.ERR_UNSUPPORTED and "1024" in msg
    assert _status(sm, "big", NoSelect, [Count("id")], ["state"])[0] == L.ERR_STATE        # count reads nothing: the dense path
