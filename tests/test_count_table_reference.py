"""The plain reference of tests/table_reference.py against the oracle and the host report, and its generator.  CPU only.

The GPU tests of the count table, its export, the union and the report filter (test_gpu_count_table.py) compare the
device with this reference; these tests pin the reference itself: its key functions equal the oracle's, and on rows
built to sit on the threshold its filter rule keeps everything the report of a one-file run can show."""
import os
import random
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import table_reference as ref   # noqa: E402
from oracle.oracle import Oracle   # noqa: E402
from trew_b200 import api   # noqa: E402


def report_text(min_mer, tables):
    rep = api.Report(min_mer)
    rep.add_file("F", tables)
    return rep.finish()


def test_key_functions_equal_the_oracle():
    o = Oracle(3, 64)
    rng = random.Random(5)
    for k in range(3, 65):
        keys = [0, (1 << (2 * k)) - 1] + [rng.getrandbits(2 * k) for _ in range(40)]
        for w in keys:
            assert ref.canon(w, k) == o.canon(w, k), (k, w)
            assert ref.canon(ref.rc(w, k), k) == o.crc(w, k), (k, w)
            assert ref.fold(w, k) == min(o.crc(o.canon(w, k), k), o.canon(w, k)), (k, w)
            assert ref.rc(ref.rc(w, k), k) == w


def test_union_and_order():
    a = [(0, 5, 7, 2 ** 32 - 1), (1, 5, 7, 1), (0, 64, (1 << 127) | 3, 2 ** 40)]
    b = [(0, 5, 7, 1), (0, 64, (1 << 127) | 3, 2 ** 40)]
    u = ref.union([a, ref.to_array(b)])
    assert u == {(0, 5, 7): 2 ** 32, (1, 5, 7): 1, (0, 64, (1 << 127) | 3): 2 ** 41}
    rows = ref.sorted_rows({(0, 5, 1 << 64): 1, (0, 5, (1 << 63)): 1, (0, 4, 9): 1, (1, 3, 0): 1})
    assert [r[:3] for r in rows] == [(0, 4, 9), (0, 5, 1 << 63), (0, 5, 1 << 64), (1, 3, 0)]
    arr = ref.to_array(rows)
    assert arr[1, 0] < 0                         # seq_lo with bit 63 set is negative as int64
    assert ref.from_array(arr) == rows


@pytest.mark.parametrize("mx", [32, 64])
def test_generator_is_deterministic_and_covers_the_edges(mx):
    a, b = ref.edge_rows(3, mx), ref.edge_rows(3, mx)
    assert a == b and a != ref.edge_rows(4, mx)
    keys = {(tb, k, s) for tb, k, s, _ in a}
    assert len(keys) == len(a)
    ks = {k for _, k, _, _ in a}
    assert {3, 31, 32} <= ks and ({33, 64} <= ks) == (mx == 64) and max(ks) == mx
    assert any(s >> 63 & 1 and s < 1 << 64 for _, _, s, _ in a)
    assert any(s >> 64 for _, _, s, _ in a) == (mx > 32)
    assert {1, 2 ** 32 - 1, 2 ** 32, 2 ** 40} <= {c for _, _, _, c in a}
    # keys that differ in exactly one of table, k, seq_hi, seq_lo
    by_seq = {}
    for tb, k, s in keys:
        by_seq.setdefault(s, set()).add((tb, k))
    assert sum(1 for tb, k, s in keys if any(t2 != tb and k2 == k for t2, k2 in by_seq[s])) > 50
    assert sum(1 for tb, k, s in keys if any(t2 == tb and k2 != k for t2, k2 in by_seq[s])) > 50
    lo_twins = sum(1 for tb, k, s in keys for b in range(64) if (tb, k, s ^ (1 << b)) in keys)
    assert lo_twins > 50
    if mx > 32:
        hi_twins = sum(1 for tb, k, s in keys if k > 32 for b in range(64, 2 * k) if (tb, k, s ^ (1 << b)) in keys)
        assert hi_twins > 20
    g1, g2 = ref.report_groups(1, mx, 10), ref.report_groups(1, mx, 10)
    assert g1 == g2


@pytest.mark.parametrize("m", [1, 10, 1000, 2 ** 31, 3_000_000_000, 2 ** 32 - 1])
def test_report_groups_sit_on_the_threshold(m):
    rows = ref.report_groups(2, 64, m)
    keys = [(tb, k, s) for tb, k, s, _ in rows]
    assert len(set(keys)) == len(keys)
    tables = ref.union([rows])
    tot = ref.group_totals(tables)
    highest = [max(t) for t in tot.values()]
    if m > 1:
        assert m - 1 in highest
    assert m in highest and m + 1 in highest
    clamped = [sum(min(c, m) for (tb, k, s), c in tables.items() if (k, ref.fold(s, k)) == g and tb & 1 == cls)
               for g, t in tot.items() for cls in (0, 1) if t[cls] > 2 * m]
    assert clamped and max(clamped) >= 2 * m   # groups whose clamped class sums pass 2^32 for m >= 2^31
    assert any(s == ref.canon(ref.rc(s, k), k) for _, k, s, _ in rows)            # palindromic units
    assert any(tb >= 4 and s != ref.canon(s, k) for tb, k, s, _ in rows)            # non-canonical 'both' rows
    assert any(t[0] and t[1] and min(t) <= 3 for t in tot.values())                 # twins in the other class
    kept = ref.filter_rule(tables, m)
    assert 0 < len(kept) < len(tables) or (m == 1 and kept == tables)


@pytest.mark.parametrize("mx", [32, 64])
def test_filter_rule_keeps_what_the_report_shows(mx):
    """On report-shaped groups at the report's threshold (10) the rows the filter rule keeps give the same report text
    as all rows; dropping one kept group changes the text, so the comparison can fail."""
    mn = 5 if mx == 32 else 3
    rows = []
    for seed in range(3):
        rows += ref.report_groups(10 + seed, mx, 10)
    full = ref.union([rows])
    kept = ref.filter_rule(full, 10)
    assert len(kept) < len(full)
    text = report_text(mn, full)
    assert text.count("\n") > 20
    assert report_text(mn, kept) == text
    tot = ref.group_totals(kept)
    top = max(tot, key=lambda g: (max(tot[g]), g))
    less = {key: c for key, c in kept.items() if (key[1], ref.fold(key[2], key[1])) != top}
    assert report_text(mn, less) != text
