"""An independent evaluation of a select tree for the real-OR tests: the And / Or / Select / NoSelect tree is walked directly
with numpy over a table's rows in canonical order, without expanding it to disjunctive normal form (select_dnf).  A leaf
means what the oracle's SelectOp means: the number is narrowed with orc_d2i (INT) / orc_d2b (TINYINT) and compared
strictly; a Match literal of another length than the column's width matches nothing.

Also here: the planner's narrowing of one conjunction, restated (`can_hold`: does a conjunction survive narrowing, or is
it dropped from a disjunction before any kernel runs), and a seeded generator of random select trees."""
from __future__ import annotations

import numpy as np

import oracle_lib as O
from immutable3_b200 import And, EQ, GT, LT, Match, NoSelect, Or, Select
from immutable3_b200.engine import MAX_OR_TERMS


def canonical_columns(orc, table, names):
    """{name: column} of every row of the table in canonical order (valid for any segment count)."""
    res = orc.query(table, [], list(names))
    return dict(zip(names, res.columns))


def _number(col, v):
    return int(O.lib().orc_d2i(float(v))) if col.dtype == np.int32 else int(O.lib().orc_d2b(float(v)))


def leaf_mask(col, cond):
    if isinstance(cond, Match):
        w = col.dtype.itemsize
        lits = [v.encode() for v in cond.values if len(v.encode()) == w]
        return np.isin(col, np.array(lits, dtype=col.dtype)) if lits else np.zeros(len(col), bool)
    c = col.astype(np.int64)
    if isinstance(cond, GT):
        return c > _number(col, cond.gt)
    if isinstance(cond, LT):
        return c < _number(col, cond.lt)
    if isinstance(cond, EQ):
        return c == _number(col, cond.eq)
    raise TypeError(f"not a supported condition: {cond!r}")


def eval_tree(cols, select):
    """Bool mask of the rows (canonical order) the select tree holds on."""
    n = len(next(iter(cols.values())))
    if isinstance(select, Or):
        return eval_tree(cols, select.op1) | eval_tree(cols, select.op2)
    if isinstance(select, And):
        return eval_tree(cols, select.op1) & eval_tree(cols, select.op2)
    if isinstance(select, Select):
        return leaf_mask(cols[select.col], select.cond)
    if select is NoSelect:
        return np.ones(n, bool)
    raise TypeError(f"not a select tree: {select!r}")


def expected_rows(cols, mask, proj, limit=0):
    """The projected columns of the selected rows, cut at LIMIT (0 = no LIMIT) in canonical order."""
    idx = np.flatnonzero(mask)
    if limit > 0:
        idx = idx[:limit]
    return [cols[p][idx] for p in proj]


def can_hold(term, cols):
    """False if narrowing alone shows the conjunction (a list of leaves) never holds: an empty range on a numeric column, or
    no literal of the column's width common to its Match lists.  Such a term is dropped from a disjunction."""
    ranges, lits = {}, {}
    for leaf in term:
        col, cond = cols[leaf.col], leaf.cond
        if isinstance(cond, Match):
            mine = {v.encode() for v in cond.values if len(v.encode()) == col.dtype.itemsize}
            lits[leaf.col] = mine if leaf.col not in lits else lits[leaf.col] & mine
            continue
        lo, hi = ranges.get(leaf.col, (-2**31, 2**31 - 1) if col.dtype == np.int32 else (-128, 127))
        if isinstance(cond, GT):
            lo = max(lo, _number(col, cond.gt) + 1)
        elif isinstance(cond, LT):
            hi = min(hi, _number(col, cond.lt) - 1)
        else:
            k = _number(col, cond.eq)
            lo, hi = max(lo, k), min(hi, k)
        ranges[leaf.col] = (lo, hi)
    return all(lo <= hi for lo, hi in ranges.values()) and all(lits.values())


def dnf_size(select):
    """Number of conjunctions the tree expands to, without expanding it."""
    if isinstance(select, Or):
        return dnf_size(select.op1) + dnf_size(select.op2)
    if isinstance(select, And):
        return dnf_size(select.op1) * dnf_size(select.op2)
    return 1


def random_tree(rng, leaf, depth=3, max_terms=MAX_OR_TERMS):
    """A random And / Or tree of depth <= `depth` over leaves drawn by `leaf(rng)`, expanding to at most `max_terms`
    conjunctions."""
    def grow(d):
        if d == 0 or rng.random() < 0.3:
            return leaf(rng)
        op = And if rng.random() < 0.5 else Or
        return op(grow(d - 1), grow(d - 1))

    while True:
        t = grow(depth)
        if dnf_size(t) <= max_terms:
            return t
