"""Reference for Sum / Avg aggregates (imm3_query_agg_ext), restated from the oracle's selected rows.

The oracle's C restatement (oracle/oracle.c) resolves only Count / Min / Max, as the reference engine does.  Here the
oracle's row query supplies the selected rows in canonical order, and numpy groups them in first-appearance order:
Count = the group's rows, Min / Max = the extremes as float64, Sum = the exact int64 sum, Avg = float64(sum) /
float64(count).  The Count / Min / Max part, and the group order, are checked against the oracle's own query_agg, so the
grouping here is the oracle's."""
import numpy as np

import oracle_lib as O
from helpers import oracle_preds
from immutable3_b200 import Avg, Count, Max, Min, Sum

_ORC_OPS = {Count: O.AGG_COUNT, Min: O.AGG_MIN, Max: O.AGG_MAX}


def group_rows(keys, n):
    """keys: list of n-long arrays -> (inverse group index per row in first-appearance order, first row of each group)."""
    if not keys:
        inv = np.zeros(n, np.int64)
        return inv, (np.zeros(1, np.int64) if n else np.zeros(0, np.int64))
    code = np.zeros(n, np.int64)
    for k in keys:
        u, ki = np.unique(k, return_inverse=True)
        code = code * len(u) + ki.reshape(-1)
    u, first, inv = np.unique(code, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")        # groups by first appearance
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    return rank[inv.reshape(-1)], first[order]


def sum_avg_columns(keys, values, aggs):
    """Group columns then one column per aggregate for rows given as `keys` (group columns) and `values` (col -> array)."""
    inv, first = group_rows(keys, len(next(iter(values.values()))))
    ng = len(first)
    cnt = np.bincount(inv, minlength=ng).astype(np.int64)
    out = [k[first] for k in keys]
    for a in aggs:
        v = values[a.col]
        if isinstance(a, Count):
            out.append(cnt)
        elif isinstance(a, (Sum, Avg)):
            s = np.zeros(ng, np.int64)
            np.add.at(s, inv, v.astype(np.int64))
            out.append(s if isinstance(a, Sum) else s.astype(np.float64) / cnt.astype(np.float64))
        else:
            m = np.full(ng, np.iinfo(np.int64).max if isinstance(a, Min) else np.iinfo(np.int64).min, np.int64)
            (np.minimum if isinstance(a, Min) else np.maximum).at(m, inv, v.astype(np.int64))
            out.append(m.astype(np.float64))
    return out


def query_agg_ext(orc, table, sel, aggs, group_by, seg_begin=0, seg_end=-1):
    """The expected columns of imm3_query_agg_ext over the oracle's rows (segments [seg_begin, seg_end))."""
    group_by = list(group_by)
    cols = list(dict.fromkeys(group_by + [a.col for a in aggs]))
    rows = orc.query(table, oracle_preds(sel), cols, limit=0, seg_begin=seg_begin, seg_end=seg_end)
    data = {c: (np.asarray(rows.columns[i]) if rows.columns else np.empty(0)) for i, c in enumerate(cols)}
    n = len(data[cols[0]]) if rows.columns else 0
    keys = [data[g] for g in group_by]
    exp = sum_avg_columns(keys, data, aggs) if n else [np.empty(0)] * (len(group_by) + len(aggs))
    # the oracle's own Count / Min / Max over the same query: group order and values must agree
    plain = [a for a in aggs if type(a) in _ORC_OPS] or [Count(aggs[0].col)]
    ref = orc.query_agg(table, oracle_preds(sel), [(_ORC_OPS[type(a)], a.col) for a in plain], group_by, seg_begin=seg_begin, seg_end=seg_end)
    assert ref.nrows == (len(exp[0]) if n else 0), (ref.nrows, n)
    if n:
        for g in range(len(group_by)):
            assert np.array_equal(ref.columns[g], exp[g])
        mine = sum_avg_columns(keys, data, plain)
        for c in range(len(plain)):
            assert np.array_equal(ref.columns[len(group_by) + c], mine[len(group_by) + c])
    return exp


def java_double(v: float) -> str:
    """Double.toString with the shortest round-trip digits (Python's repr digits)."""
    if v != v:
        return "NaN"
    if v in (float("inf"), float("-inf")):
        return "Infinity" if v > 0 else "-Infinity"
    if v == 0:
        return "-0.0" if str(v).startswith("-") else "0.0"
    sign = "-" if v < 0 else ""
    a = abs(v)
    digits, e10 = _digits(a)
    if 1e-3 <= a < 1e7:
        if e10 < 0:
            return sign + "0." + "0" * (-e10 - 1) + digits
        ip = digits[:e10 + 1].ljust(e10 + 1, "0")
        return sign + ip + "." + (digits[e10 + 1:] or "0")
    return sign + digits[0] + "." + (digits[1:] or "0") + "E" + str(e10)


def _digits(a: float):
    """(significant digits, decimal exponent of the first one) of repr(a)."""
    r = repr(a)
    if "e" in r:
        mant, ex = r.split("e")
        ex = int(ex)
    else:
        mant, ex = r, 0
    if "." in mant:
        ip, fp = mant.split(".")
    else:
        ip, fp = mant, ""
    fp = fp.rstrip("0") if fp != "0" else ""
    allds = (ip + fp).lstrip("0")
    lead = len(ip.lstrip("0"))
    if lead:
        e10 = lead - 1 + ex
    else:
        e10 = -(len(fp) - len(fp.lstrip("0"))) - 1 + ex
    return allds.rstrip("0") or "0", e10
