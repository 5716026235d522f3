"""Plain reference of the device count table and its export, union and report filter, plus a seeded generator of
constructed rows.  TEST INFRASTRUCTURE ONLY.

Everything here is Python integers: keys are 128-bit `seq` values, counts are unbounded, and numpy is only used to
lay rows out (or read them back) in trew_entry layout, never to compute on keys.

Rows are (table, k, seq, count) tuples; tables are {(table, k, seq): count} dicts (the layout DeviceContext.finish()
returns).  As a (n, 4) int64 array a row is one trew_entry: seq_lo, seq_hi, count, table | k << 32.
"""
import random
from typing import Dict, Iterable, List, Sequence, Tuple

import numpy as np

Row = Tuple[int, int, int, int]
Tables = Dict[Tuple[int, int, int], int]

M64 = (1 << 64) - 1


# ---- rows <-> trew_entry arrays ---------------------------------------------------------------------------------------

def to_array(rows: Sequence[Row]) -> np.ndarray:
    """Rows -> (n, 4) int64 array in trew_entry layout (64-bit fields reinterpreted as signed)."""
    out = np.zeros((len(rows), 4), dtype=np.uint64)
    if rows:
        out[:] = [(seq & M64, seq >> 64, c, tb | (k << 32)) for tb, k, seq, c in rows]
    return out.view(np.int64)


def from_array(a: np.ndarray) -> List[Row]:
    """(n, 4) int64 array in trew_entry layout -> rows."""
    return [(m & 0xffffffff, m >> 32, (hi << 64) | lo, c)
            for lo, hi, c, m in np.ascontiguousarray(a).view(np.uint64).reshape(-1, 4).tolist()]


def from_view(v: np.ndarray) -> List[Row]:
    """A structured entry array (DeviceContext.ENTRY_DTYPE, e.g. finish_view()) -> rows, order kept."""
    return list(zip(v["table"].tolist(), v["k"].tolist(),
                    [(hi << 64) | lo for lo, hi in zip(v["seq_lo"].tolist(), v["seq_hi"].tolist())], v["count"].tolist()))


def rows_of(tables: Tables) -> List[Row]:
    return [(tb, k, seq, c) for (tb, k, seq), c in tables.items()]


# ---- the reference ----------------------------------------------------------------------------------------------------

def union(lists: Iterable) -> Tables:
    """Sum of several row lists (each a list of rows, a (n, 4) entry array or a tables dict), keyed by (table, k, seq)."""
    out: Tables = {}
    for rows in lists:
        if isinstance(rows, np.ndarray):
            rows = from_array(rows)
        elif isinstance(rows, dict):
            rows = rows_of(rows)
        for tb, k, seq, c in rows:
            key = (tb, k, seq)
            out[key] = out.get(key, 0) + c
    return out


def scaled(tables: Tables, times: int) -> Tables:
    return {key: c * times for key, c in tables.items()}


def sorted_rows(tables: Tables) -> List[Row]:
    """The rows in export order: (table, k, seq_hi, seq_lo), all unsigned -- which is (table, k, seq)."""
    return [(tb, k, seq, c) for (tb, k, seq), c in sorted(tables.items())]


def canon(w: int, k: int) -> int:
    """Smallest rotation of the k-base key w (2 bits per base)."""
    mask = (1 << (2 * k)) - 1
    best, cur = w, w
    for _ in range(k - 1):
        cur = ((cur & 3) << (2 * (k - 1))) | (cur >> 2)
        best = min(best, cur & mask)
    return best


def rc(w: int, k: int) -> int:
    """Reverse complement (codes T G C A = 0 1 2 3, so the complement of x is 3 - x)."""
    r = 0
    for _ in range(k):
        r = (r << 2) | (3 - (w & 3))
        w >>= 2
    return r


def fold(w: int, k: int) -> int:
    """The report's group of a key: min(canonical rotation of the reverse complement, canonical rotation)."""
    return min(canon(rc(w, k), k), canon(w, k))


def group_totals(tables: Tables) -> Dict[Tuple[int, int], List[int]]:
    """{(k, fold): [high-class total, low-class total]} (the class is table & 1)."""
    tot: Dict[Tuple[int, int], List[int]] = {}
    for (tb, k, seq), c in tables.items():
        tot.setdefault((k, fold(seq, k)), [0, 0])[tb & 1] += c
    return tot


def filter_rule(tables: Tables, min_total: int) -> Tables:
    """Every row of a (k, fold) group whose high-class or low-class total is >= min_total."""
    tot = group_totals(tables)
    return {key: c for key, c in tables.items() if max(tot[(key[1], fold(key[2], key[1]))]) >= min_total}


# ---- the generator ----------------------------------------------------------------------------------------------------

BIG_COUNTS = (1, 2 ** 32 - 1, 2 ** 32, 2 ** 40)


def _key(rng: random.Random, k: int) -> int:
    return rng.getrandbits(2 * k)


def _ks(max_mer: int) -> List[int]:
    edges = [3, 31, 32, 33, 64]
    return [k for k in edges if k <= max_mer] + list(range(3, max_mer + 1))


def edge_rows(seed: int, max_mer: int, n_random: int = 400) -> List[Row]:
    """Distinct keys at the edges a table, a sort or a union can get wrong: seq 0 (all T) and the all-A key at every k
    of the list, k = 3 / 31 / 32 / 33 / 64 where max_mer allows, seq_lo with bit 63 set, seq_hi != 0 only when
    max_mer > 32, pairs of keys that differ in exactly one of table, k, seq_hi and seq_lo; counts 1, 2^32 - 1, 2^32,
    2^40 and random."""
    rng = random.Random(seed)
    ks = sorted(set(_ks(max_mer)))
    out: Dict[Tuple[int, int, int], int] = {}

    def count():
        return rng.choice(BIG_COUNTS) if rng.random() < 0.5 else rng.randint(1, 1000)

    def put(tb, k, seq):
        assert 0 <= seq < 1 << (2 * k)
        out.setdefault((tb, k, seq), count())

    for k in ks:
        for tb in range(6):
            put(tb, k, 0)                               # all T
            put(tb, k, (1 << (2 * k)) - 1)              # all A
        if k >= 32:
            put(rng.randrange(6), k, (1 << 63) | _key(rng, 31))   # seq_lo negative as int64, seq_hi 0
        if k > 32:
            put(rng.randrange(6), k, (1 << 127 if k == 64 else 0) | (1 << 63) | _key(rng, k) >> 2 << 2)
    for _ in range(n_random):
        k = rng.choice(ks)
        tb = rng.randrange(6)
        seq = _key(rng, k)
        put(tb, k, seq)
        # twins that differ in exactly one field
        put((tb + 1 + rng.randrange(5)) % 6, k, seq)
        k2 = rng.choice([x for x in ks if x != k and seq < 1 << (2 * x)] or [k])
        put(tb, k2, seq)
        if k > 32:
            put(tb, k, seq ^ (1 << (64 + rng.randrange(2 * k - 64))))   # seq_hi differs
        put(tb, k, seq ^ (1 << rng.randrange(min(64, 2 * k))))             # seq_lo differs
    return [(tb, k, seq, c) for (tb, k, seq), c in out.items()]


def split(rng: random.Random, total: int, parts: int) -> List[int]:
    """total as `parts` positive integers (parts <= total)."""
    cuts = sorted(rng.sample(range(1, total), parts - 1)) if parts > 1 and total < 1 << 20 else \
        sorted({rng.randrange(1, total) for _ in range(parts - 1)})
    bounds = [0] + cuts + [total]
    return [b - a for a, b in zip(bounds, bounds[1:])]


def _palindrome(rng: random.Random, k: int) -> int:
    """A key whose reverse complement is itself (k even): u followed by rc(u)."""
    h = k // 2
    u = _key(rng, h)
    return (u << (2 * h)) | rc(u, h)


def _candidates(c: int, t: int, k: int, cls: int) -> List[Tuple[int, int]]:
    """(table, key) slots of one class of the group of canonical rotations c and t = canon(rc(c)): forward and backward
    rows hold c or t; 'both' rows any rotation of either strand (the large-k path leaves them non-canonical)."""
    out = []
    for base in (0, 1):
        for key in sorted({c, t}):
            out.append((2 * base + cls, key))
    rots = set()
    for w in (c, rc(c, k)):
        cur = w
        for _ in range(k):
            rots.add(cur)
            cur = ((cur & 3) << (2 * (k - 1))) | (cur >> 2)
    out += [(4 + cls, key) for key in sorted(rots)]
    return out


def report_groups(seed: int, max_mer: int, min_total: int, n_groups: int = 240) -> List[Row]:
    """Rows shaped like the report's groups (k, fold), built to sit on min_total: one class of each group totals
    min_total - 1, min_total or min_total + 1 over 1 to 12 rows, or holds 2 to 12 rows of at least min_total each (the
    clamped sums of such a group pass 2^32 when min_total >= 2^31); some groups are palindromic (crc(seq) == seq), some
    get twins in the other class with small counts.  Distinct groups, distinct keys."""
    rng = random.Random(seed * 1_000_003 + min_total)
    ks = sorted(set(_ks(max_mer)))
    used = set()
    out: List[Row] = []
    for g in range(n_groups):
        for _ in range(100):
            k = rng.choice(ks)
            w = _palindrome(rng, k) if g % 7 == 3 and k % 2 == 0 else _key(rng, k)
            c = canon(w, k)
            if (k, fold(c, k)) not in used:
                break
        else:
            continue
        used.add((k, fold(c, k)))
        t = canon(rc(c, k), k)
        cls = rng.randrange(2)
        slots = _candidates(c, t, k, cls)
        rng.shuffle(slots)
        kind = g % 4
        if kind == 3:   # heavy: every row at least min_total
            n = rng.randint(2, min(12, len(slots)))
            counts = [rng.choice([min_total, min_total + 1, max(min_total, 3_000_000_000), max(min_total, 2 ** 32), 2 ** 40])
                      for _ in range(n)]
        else:
            total = min_total - 1 + kind   # kind 0 / 1 / 2: one below, at, one above
            if total <= 0:
                total = 1
            n = rng.randint(1, min(12, len(slots), total))
            counts = split(rng, total, n)
        out += [(tb, k, key, cnt) for (tb, key), cnt in zip(slots, counts)]
        if rng.random() < 0.4:   # twins in the other class, small counts
            other = _candidates(c, t, k, 1 - cls)
            for tb, key in rng.sample(other, rng.randint(1, min(3, len(other)))):
                out.append((tb, k, key, rng.randint(1, 3)))
    return out
