"""Exact numpy group-by in first-appearance order, and restatements of the aggregation kernels' key packing and hashes
(k_agg.cuh), for tests of group order and group keys.

* `group_by` aggregates canonical-order arrays the way ProjectAggOp reports them with one worker: one row per group in the
  order of the group's first row, the group cells of that row, COUNT / SUM as int64, MIN / MAX of the raw int32 / int8
  values as float64, AVG as float64(sum) / float64(count).  It never uses helpers.numpy_expected, which assumes that
  canonical order is write order.
* `pack_keys` is the kernels' key: the group cells little-endian at key_shift = 8 x the widths of the cells before them
  (a TINYINT cell is its raw byte, an INT cell its four bytes, byte b of a STRING(k) cell sits at bit 8b).
* `agg_hash32`, `agg_hash`, `cta_home`, `guess_index` and `global_home` restate the hashes of the CTA key table, its guess
  cache and the global table; they only serve to construct adversarial key sets (tests/test_agg_hash_host.py pins their
  constants to the kernel source).
"""
import numpy as np

from immutable3_b200 import Avg, Count, Max, Min, Sum

# k_agg.cuh: agg_hash32's two multipliers, agg_hash's multiplier, the CTA table and its guess cache
HASH32_MUL_LO = 0x9E3779B1
HASH32_MUL_HI = 0x85EBCA6B
HASH64_MUL = 0xFF51AFD7ED558CCD
CTA_SLOTS = 256        # kAggSlots
DICT_BITS = 14         # kAggDictBits
CTA_PROBES = 16        # agg_cta_slot's probe bound
GLOBAL_SLOTS = 1 << 16  # the global table without IMM3_AGG_SLOTS

_M32 = np.uint64(0xFFFFFFFF)


def agg_hash32(keys):
    """((uint32)k * 0x9E3779B1) ^ ((uint32)(k >> 32) * 0x85EBCA6B), elementwise on uint64 keys -> uint64 in [0, 2^32)."""
    k = np.asarray(keys, dtype=np.uint64)
    lo = ((k & _M32) * np.uint64(HASH32_MUL_LO)) & _M32
    hi = ((k >> np.uint64(32)) * np.uint64(HASH32_MUL_HI)) & _M32
    return lo ^ hi


def agg_hash(keys):
    """k ^= k >> 33; k *= 0xFF51AFD7ED558CCD (mod 2^64); k ^= k >> 33; low 32 bits."""
    k = np.asarray(keys, dtype=np.uint64)
    k = k ^ (k >> np.uint64(33))
    with np.errstate(over="ignore"):
        k = k * np.uint64(HASH64_MUL)
    k = k ^ (k >> np.uint64(33))
    return k & _M32


def cta_home(keys):
    """First slot agg_cta_slot probes: hh >> 24."""
    return agg_hash32(keys) >> np.uint64(24)


def guess_index(keys):
    """Entry of the hash -> slot cache: hh >> (32 - kAggDictBits)."""
    return agg_hash32(keys) >> np.uint64(32 - DICT_BITS)


def global_home(keys, slots):
    """First slot agg_global_slot probes in a table of `slots` entries."""
    return agg_hash(keys) & np.uint64(slots - 1)


def cell_bytes(col):
    """[n, width] uint8 view of a column's cells as the kernels read them (INT little-endian, TINYINT raw, STRING raw)."""
    a = np.ascontiguousarray(col)
    return a.view(np.uint8).reshape(len(a), a.dtype.itemsize)


def pack_keys(cols):
    """The packed 64-bit group key of every row (uint64); at most 7 key bytes, as the planner allows."""
    n = len(cols[0]) if cols else 0
    if not cols:
        return np.zeros(n, np.uint64)
    b = np.concatenate([cell_bytes(c) for c in cols], axis=1)
    assert b.shape[1] <= 7, "group-by cells must pack into 7 bytes"
    out = np.zeros((n, 8), np.uint8)
    out[:, :b.shape[1]] = b
    return out.view("<u8").reshape(n)


def int_keys(values):
    """Packed key of an INT group column alone (its four bytes, zero-extended)."""
    return np.asarray(values, dtype=np.int32).view(np.uint32).astype(np.uint64)


def canonical_segment_order(nsegments):
    """Write-order segment indices in canonical order: the file names' lexicographic order (0, 1, 10, 11, 2, ...)."""
    return sorted(range(nsegments), key=str)


def write_order(cols, nrows, block_size, segment_size):
    """Arrays meant in CANONICAL order -> the same rows in write order (what SegmentWriter must be given)."""
    per = block_size * segment_size + 1
    nseg = (nrows + per - 1) // per
    lens = [min(per, nrows - s * per) for s in range(nseg)]
    start, pos = {}, 0
    for s in canonical_segment_order(nseg):
        start[s] = pos
        pos += lens[s]
    idx = np.concatenate([np.arange(start[s], start[s] + lens[s]) for s in range(nseg)]) if nseg else np.zeros(0, np.int64)
    done = {}  # (twin columns naming one array are permuted once)
    for v in cols.values():
        if id(v) not in done:
            done[id(v)] = v[idx]
    return {k: done[id(v)] for k, v in cols.items()}


class Groups:
    """Rows of `keys` (canonical order, selected rows only) grouped in first-appearance order."""

    def __init__(self, key_cols, n):
        self.n = n
        if n == 0:
            self.ngroups, self.first = 0, np.zeros(0, np.int64)
            return
        if not key_cols:
            self.ngroups, self.first = 1, np.zeros(1, np.int64)
            self.perm, self.starts = np.arange(n), np.zeros(1, np.int64)
            return
        packed = pack_keys(key_cols)
        self.perm = np.argsort(packed, kind="stable")               # equal keys keep row order: the first is the group's first row
        sk = packed[self.perm]
        self.starts = np.flatnonzero(np.concatenate(([True], sk[1:] != sk[:-1])))
        first_sorted = self.perm[self.starts]
        order = np.argsort(first_sorted, kind="stable")             # groups by first row
        self.ngroups = len(self.starts)
        self.first = first_sorted[order]
        self.order = order

    def _per_group(self, reduced):
        """Per-group values in key order -> first-appearance order."""
        return reduced if not hasattr(self, "order") else reduced[self.order]

    def cells(self, col):
        return np.asarray(col)[self.first]

    def count(self):
        ends = np.concatenate((self.starts[1:], [self.n]))
        return self._per_group((ends - self.starts).astype(np.int64))

    def reduce(self, ufunc, values):
        v = np.asarray(values).astype(np.int64)[self.perm]
        return self._per_group(ufunc.reduceat(v, self.starts))


def group_by(key_cols, values, aggs, groups=None):
    """Expected result columns of ProjectAgg(aggs, group_by) over selected canonical-order rows: the group cells, then one
    column per aggregate.  key_cols: the group columns' arrays; values: column name -> array; groups: the Groups of these
    rows when the caller has them (the same grouping under other key columns that are functions of each other)."""
    n = len(key_cols[0]) if key_cols else len(next(iter(values.values())))
    g = groups if groups is not None else Groups(key_cols, n)
    assert g.n == n
    if g.ngroups == 0:
        return [np.empty(0, np.asarray(c).dtype) for c in key_cols] + [np.empty(0) for _ in aggs]
    out = [g.cells(c) for c in key_cols]
    cnt = g.count()
    for a in aggs:
        if isinstance(a, Count):
            out.append(cnt)
        elif isinstance(a, (Sum, Avg)):
            s = g.reduce(np.add, values[a.col])
            out.append(s if isinstance(a, Sum) else s.astype(np.float64) / cnt.astype(np.float64))
        else:
            out.append(g.reduce(np.minimum if isinstance(a, Min) else np.maximum, values[a.col]).astype(np.float64))
    return out


# ---- adversarial key sets ------------------------------------------------------------------------------------------------

def int_keys_with_cta_home(home, count, rng, exclude=()):
    """`count` distinct int32 values whose INT key has CTA home `home`."""
    out = []
    seen = set(int(x) for x in exclude)
    while len(out) < count:
        cand = rng.integers(-2**31, 2**31, 1 << 16, dtype=np.int64).astype(np.int32)
        for v in cand[cta_home(int_keys(cand)) == np.uint64(home)]:
            if int(v) not in seen:
                seen.add(int(v))
                out.append(int(v))
    return np.array(out[:count], np.int32)


def int_keys_with_guess(index, count, rng):
    """`count` distinct int32 values whose INT key has guess-cache entry `index` (and so one CTA home)."""
    inv = pow(HASH32_MUL_LO, -1, 1 << 32)
    x = (np.uint64(index) << np.uint64(32 - DICT_BITS)) + rng.choice(1 << (32 - DICT_BITS), count, replace=False).astype(np.uint64)
    k = (x * np.uint64(inv)) & _M32                                  # hh = k * A mod 2^32 for keys below 2^32
    return k.astype(np.uint32).view(np.int32)


def high_words_sharing_guess(count, rng, bits=24):
    """`count` distinct values h < 2^bits whose (h * 0x85EBCA6B mod 2^32) share their top kAggDictBits bits: 7-byte keys
    with equal low 32 bits and these high bits share the guess-cache entry."""
    h = rng.choice(1 << bits, 1 << 17, replace=False).astype(np.uint64)
    top = ((h * np.uint64(HASH32_MUL_HI)) & _M32) >> np.uint64(32 - DICT_BITS)
    vals, inv, cnt = np.unique(top, return_inverse=True, return_counts=True)
    best = int(np.argmax(cnt))
    assert cnt[best] >= count, cnt[best]
    return np.sort(h[inv.reshape(-1) == best][:count])


def int_keys_with_global_home(home, slots, count, rng, exclude=()):
    """`count` distinct int32 values whose INT key has home `home` in a global table of `slots` entries."""
    out = []
    seen = set(int(x) for x in exclude)
    while len(out) < count:
        cand = rng.integers(-2**31, 2**31, 1 << 16, dtype=np.int64).astype(np.int32)
        for v in cand[global_home(int_keys(cand), slots) == np.uint64(home)]:
            if int(v) not in seen:
                seen.add(int(v))
                out.append(int(v))
    return np.array(out[:count], np.int32)


SMALL_SLOTS = 64        # IMM3_AGG_SLOTS of the full-table cases
CTA_HOME = 77           # the CTA home the hot keys share
WRAP_HOME = 60          # the global home of the full-table keys: their probe sequence wraps past slot 63


def adversarial_keys(seed=1234):
    """The key sets of the adversarial aggregation tests (tests/test_gpu_agg_order_keys.py), each with the property
    tests/test_agg_hash_host.py checks:
      hot     24 INT keys with one CTA home (more than the 16 slots agg_cta_slot probes), of 44 groups in all (`cta`)
      guess4  6 INT keys with one guess-cache entry
      pairs   (INT, STRING(3)) groups packed into 7-byte keys: 6 with the same INT cell (equal low 32 bits) and high bytes
              that share the guess-cache entry, then the guess4 keys with an all-0x00 cell, then 8 random pairs
      full64  64 INT keys with one home in a 64-slot global table, at slot 60: the probe sequence wraps past slot 63
      over65  full64 and one more key: one group more than the table holds"""
    rng = np.random.default_rng(seed)
    hot = int_keys_with_cta_home(CTA_HOME, 24, rng)
    others = rng.choice(np.arange(-2**31, 2**31 - 1, 1 << 12, dtype=np.int64), 40, replace=False).astype(np.int32)
    others = others[cta_home(int_keys(others)) != np.uint64(CTA_HOME)][:20]
    cta = np.concatenate([hot, others])
    guess4 = int_keys_with_guess(int(rng.integers(0, 1 << DICT_BITS)), 6, rng)
    low = np.int32(rng.integers(-2**31, 2**31))
    hi7 = high_words_sharing_guess(6, rng)
    rk = rng.integers(-2**31, 2**31, 8, dtype=np.int64).astype(np.int32)
    rh = rng.integers(0, 1 << 24, 8, dtype=np.int64)
    pair_k = np.concatenate([np.full(6, low, np.int32), guess4, rk])
    pair_h = np.concatenate([hi7.astype(np.int64), np.zeros(6, np.int64), rh])
    pair_s = np.array([int(h).to_bytes(3, "little") for h in pair_h], "S3")
    full64 = int_keys_with_global_home(WRAP_HOME, SMALL_SLOTS, SMALL_SLOTS, rng)
    extra = int_keys_with_global_home((WRAP_HOME + 7) % SMALL_SLOTS, SMALL_SLOTS, 1, rng, exclude=full64)
    return {"hot": hot, "cta": cta, "guess4": guess4, "pair_k": pair_k, "pair_s": pair_s, "full64": full64,
            "over65": np.concatenate([full64, extra])}


def introduced_over_time(keys, n, rng, spacing=64):
    """n rows whose key j first appears at row j * spacing; every other row draws uniformly from the keys introduced by then."""
    k = np.asarray(keys)
    m = len(k)
    row = np.arange(n)
    avail = np.minimum(row // spacing + 1, m)
    idx = (rng.random(n) * avail).astype(np.int64)
    intro = np.arange(min(m, (n + spacing - 1) // spacing)) * spacing
    idx[intro] = np.arange(len(intro))
    return idx
