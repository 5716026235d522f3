"""The device count table and everything that turns it into rows, against the plain reference of table_reference.py:
inserts through trew_dev_merge_rows (a full table, a wrap past the last slot, one key from millions of threads at once,
an overflow, a rehash), the compaction at its first-pass capacity, the sort-based union of several row lists, and the
report filter at thresholds from 1 to 2^32 - 1.  Then the scan tables of multi-million-read batches against the oracle,
through the staging table's overflow and the direct adds, and counts past 2^32.  Every comparison is exact."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import table_reference as ref   # noqa: E402
from trew_b200 import api, synth   # noqa: E402

pytestmark = pytest.mark.gpu

CONFIGS = [(5, 32), (3, 64)]   # narrow sort (seq_lo only) and wide sort (seq_hi too)
M64 = (1 << 64) - 1


def on_device(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr)).to("cuda:0")


class _DevRows:
    """A (n, 4) int64 view of library-owned device memory, through the CUDA array interface."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n, 4), "typestr": "<i8", "data": (ptr, False), "version": 3}


def read_device_rows(ptr, n):
    import torch
    if n == 0:
        return []
    return ref.from_array(torch.as_tensor(_DevRows(ptr, n), device="cuda:0").cpu().numpy())


def check(got, want, what=""):
    """got / want: row lists; a short message instead of a diff of a million rows."""
    if got == want:
        return
    g, w = set(got), set(want)
    msg = "%s: %d rows, want %d; only device %s; only reference %s" % (what, len(got), len(want), sorted(g - w)[:4], sorted(w - g)[:4])
    if g == w:
        msg += "; same rows, order or duplicates differ"
    raise AssertionError(msg)


def finish_rows(ctx):
    return ref.from_view(ctx.finish_view())


def merged_rows(ctx, lists):
    return ref.from_view(ctx.finish_merged_view(lists))


def random_rows(seed, n, max_mer, counts=(1, 1000)):
    """n distinct keys of random (table, k) with counts in [counts[0], counts[1]]."""
    import random
    r = random.Random(seed)
    seen = set()
    out = []
    while len(out) < n:
        k = r.randint(3, max_mer)
        key = (r.randrange(6), k, r.getrandbits(2 * k))
        if key not in seen:
            seen.add(key)
            out.append(key + (r.randint(counts[0], counts[1]),))
    return out


# ---- the home slot of a key: table_add_impl's hash, restated to build probe chains on purpose -------------------------

def _mix64(x):
    x ^= x >> 33
    x = (x * 0xff51afd7ed558ccd) & M64
    x ^= x >> 33
    x = (x * 0xc4ceb9fe1a85ec53) & M64
    x ^= x >> 33
    return x


def home_slot(tb, k, seq, mask):
    meta = (tb << 8) | k
    lo, hi = seq & M64, seq >> 64
    return _mix64(lo ^ _mix64((hi + 0x9e3779b97f4a7c15 * (meta + 1)) & M64)) & mask


def keys_homing_in(seed, max_mer, first, last, n, mask=1023, avoid=()):
    """n distinct keys whose home slot in a (mask + 1)-slot table lies in [first, last]."""
    import random
    r = random.Random(seed)
    out = {}
    while len(out) < n:
        k = r.randint(3, max_mer)
        key = (r.randrange(6), k, r.getrandbits(2 * k))
        if first <= home_slot(*key, mask) <= last and key not in avoid:
            out[key] = r.randint(1, 1000)
    return [key + (c,) for key, c in out.items()]


# ---- inserts ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mn,mx", CONFIGS)
def test_full_table_from_shuffled_copies(mn, mx):
    """2^10 slots, exactly 1024 distinct keys, each in 4096 shuffled copies in one merge_rows launch: the table ends
    full, every count is 4096 times its row's (2^40 * 4096 and (2^32 - 1) * 4096 among them)."""
    edges = ref.edge_rows(21, mx, n_random=60)
    keys = {(tb, k, s) for tb, k, s, _ in edges}
    rows = (edges + [r for r in random_rows(22, 1024, mx) if r[:3] not in keys])[:1024]
    assert len(rows) == 1024
    copies = np.repeat(ref.to_array(rows), 4096, axis=0)
    copies = copies[np.random.default_rng(23).permutation(copies.shape[0])]
    want = ref.sorted_rows(ref.scaled(ref.union([rows]), 4096))
    with api.DeviceContext(api.MODE_SHORT, mn, mx, table_log2_slots=10) as ctx:
        d = on_device(copies)
        ctx.merge_rows(d.data_ptr(), d.shape[0])
        check(finish_rows(ctx), want, "full table")
        ptr, n = ctx.export_device()
        check(read_device_rows(ptr, n), want, "export_device")


@pytest.mark.parametrize("mn,mx", CONFIGS)
def test_chains_that_wrap_and_one_key_from_every_thread(mn, mx):
    """768 keys in 1024 slots without reserve (load 3/4): 40 of them have their home slot in the last 16, so at least 24
    probe chains wrap past the last slot to slot 0.  Then 4 M copies of one new key (home slot 1020, so its chain runs
    through that wrapped cluster) in one launch: every thread races to publish the same key, exactly one row results."""
    tail = keys_homing_in(31, mx, 1008, 1023, 40)
    tail_keys = {r[:3] for r in tail}
    rest = [r for r in random_rows(32, 800, mx) if r[:3] not in tail_keys][:768 - len(tail)]
    rows = tail + rest
    assert len(rows) == 768 and len({r[:3] for r in rows}) == 768
    hot = keys_homing_in(33, mx, 1020, 1020, 1, avoid={r[:3] for r in rows})[0]
    hot_rows = np.repeat(ref.to_array([hot[:3] + (1,)]), 4 << 20, axis=0)
    with api.DeviceContext(api.MODE_SHORT, mn, mx, table_log2_slots=10) as ctx:
        d = on_device(ref.to_array(rows))
        ctx.merge_rows(d.data_ptr(), d.shape[0])
        check(finish_rows(ctx), ref.sorted_rows(ref.union([rows])), "load 3/4")
        h = on_device(hot_rows)
        ctx.merge_rows(h.data_ptr(), h.shape[0])
        want = ref.union([rows, [hot[:3] + (4 << 20,)]])
        got = finish_rows(ctx)
        check(got, ref.sorted_rows(want), "one key from 4 M threads")
        assert len(got) == 769


@pytest.mark.parametrize("mn,mx", CONFIGS)
def test_overflow_is_reported_and_reset_recovers(mn, mx):
    """1025 distinct keys into 1024 slots: the adds end after one pass over the slots and finish() reports
    TREW_ERR_TABLE_FULL (a library status, not a fault); after reset() the same context counts exactly again."""
    rows = random_rows(41, 1025, mx)
    with api.DeviceContext(api.MODE_SHORT, mn, mx, table_log2_slots=10) as ctx:
        d = on_device(ref.to_array(rows))
        ctx.merge_rows(d.data_ptr(), d.shape[0])
        with pytest.raises(api.TrewError) as e:
            ctx.finish()
        assert e.value.status == 3
        ctx.reset()
        assert finish_rows(ctx) == []
        again = rows[:700]
        d2 = on_device(ref.to_array(again + again))
        ctx.merge_rows(d2.data_ptr(), d2.shape[0])
        check(finish_rows(ctx), ref.sorted_rows(ref.union([again, again])), "after reset")


@pytest.mark.parametrize("mn,mx", CONFIGS)
def test_reserve_rehashes_then_takes_300k_keys(mn, mx):
    """A 2^10-slot table with 600 keys in it, reserve(300 000) (re-inserts them into 2^21 slots), then 300 000 keys
    that overlap the first ones in one launch."""
    first = random_rows(51, 600, mx, counts=(2 ** 32 - 5, 2 ** 32 - 1))
    more = first[:200] + random_rows(52, 299_800, mx)
    with api.DeviceContext(api.MODE_SHORT, mn, mx, table_log2_slots=10) as ctx:
        d = on_device(ref.to_array(first))
        ctx.merge_rows(d.data_ptr(), d.shape[0])
        ctx.reserve(300_000)
        check(finish_rows(ctx), ref.sorted_rows(ref.union([first])), "after the rehash")
        d2 = on_device(ref.to_array(more))
        ctx.merge_rows(d2.data_ptr(), d2.shape[0])
        want = ref.union([first, more])
        assert max(want.values()) > 2 ** 32
        check(finish_rows(ctx), ref.sorted_rows(want), "300 k keys after reserve")


# ---- export -----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [0, 1, 1_310_720, 1_310_721])
def test_export_at_the_first_compaction_capacity(n):
    """The first compaction writes into 2^20 + 2^18 = 1,310,720 rows; one more key takes the count-then-grow second pass.
    Default 2^22-slot table, no reserve, fresh context per size.  finish(), export_device() and export_rows() all give
    the reference's rows; export_rows into a buffer one row short is TREW_ERR_ARG."""
    mx = 64
    rows = random_rows(60 + n % 7, n, mx, counts=(1, 2 ** 40)) if n > 1 else [(5, 64, (1 << 127) | (1 << 63), 2 ** 40)][:n]
    want = ref.sorted_rows(ref.union([rows]))
    with api.DeviceContext(api.MODE_SHORT, 3, mx) as ctx:
        if n:
            d = on_device(ref.to_array(rows))
            ctx.merge_rows(d.data_ptr(), n)
        assert ctx.export_rows() == n
        if n:
            import torch
            short = torch.zeros((max(n - 1, 1), 4), dtype=torch.int64, device="cuda:0")
            with pytest.raises(api.TrewError) as e:
                ctx.export_rows(short.data_ptr(), n - 1)
            assert e.value.status == 1
            out = torch.zeros((n, 4), dtype=torch.int64, device="cuda:0")
            assert ctx.export_rows(out.data_ptr(), n) == n
            check(sorted(ref.from_array(out.cpu().numpy())), want, "export_rows")
        ptr, m = ctx.export_device()
        assert m == n
        check(read_device_rows(ptr, m), want, "export_device")
        check(finish_rows(ctx), want, "finish")


# ---- union ------------------------------------------------------------------------------------------------------------

def assert_sorted_unique(rows):
    keys = [(tb, k, s) for tb, k, s, _ in rows]
    assert all(a < b for a, b in zip(keys, keys[1:])), "not sorted by (table, k, seq) or a key repeats"


@pytest.mark.parametrize("mn,mx", CONFIGS)
def test_union_of_lists(mn, mx):
    """finish_merged_view over [], an empty list, a single row (the one-row copy path) and four lists of 3 M rows in all
    that overlap each other and the context's own table, with repeated keys inside a list and sums past 2^32: sorted,
    no repeated key, the reference's union, and the context's own finish() unchanged afterwards."""
    import random
    with api.DeviceContext(api.MODE_SHORT, mn, mx) as ctx:
        assert merged_rows(ctx, []) == []
        empty = on_device(np.zeros((1, 4), dtype=np.int64))
        assert merged_rows(ctx, [(empty.data_ptr(), 0)]) == []
        one = [(3, mx, (1 << (2 * mx)) - 1, 2 ** 32)]
        d1 = on_device(ref.to_array(one))
        assert merged_rows(ctx, [(d1.data_ptr(), 1)]) == one

    pool = ref.edge_rows(70, mx) + random_rows(71, 400_000, mx, counts=(1, 2 ** 31))
    rng = random.Random(72)
    heavy = [r[:3] + (2 ** 32 - 1,) for r in pool[:2000]]
    own = [pool[i] for i in rng.sample(range(len(pool)), 300_000)] + heavy
    lists = []
    for j in range(4):
        idx = [rng.randrange(len(pool)) for _ in range(650_000)]   # repeats inside a list too
        lists.append([pool[i] for i in idx] + heavy)
    assert sum(map(len, lists)) + len(own) > 2_900_000
    with api.DeviceContext(api.MODE_SHORT, mn, mx) as ctx:
        d = on_device(ref.to_array(own))
        ctx.merge_rows(d.data_ptr(), d.shape[0])
        own_want = ref.sorted_rows(ref.union([own]))
        check(finish_rows(ctx), own_want, "own table")
        check(merged_rows(ctx, []), own_want, "union with no list")
        dl = [on_device(ref.to_array(x)) for x in lists]
        got = merged_rows(ctx, [(t.data_ptr(), t.shape[0]) for t in dl])
        assert_sorted_unique(got)
        want = ref.union([own] + lists)
        assert sum(1 for c in want.values() if c > 2 ** 32) >= 2000
        check(got, ref.sorted_rows(want), "union of four lists and the own table")
        check(finish_rows(ctx), own_want, "own table after the union")


# ---- report filter ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("m", [1, 9, 10, 11, 1000, 2 ** 31, 3_000_000_000, 2 ** 32 - 1])
@pytest.mark.parametrize("mn,mx", CONFIGS)
def test_report_filter_equals_the_rule(mn, mx, m):
    """set_report_filter(m) on report-shaped groups built to sit on m (table_reference.report_groups): the rows
    finish() and finish_merged_view() keep are exactly filter_rule's.  The device accumulates groups under a 64-bit
    fingerprint, and colliding groups merge (keeping more rows); with a few thousand groups here the chance of any
    collision is about 1e-8, so an exact comparison is fair.  Groups whose rows each hold at least m give class sums
    past 2^32 once m >= 2^31: totals that wrap at 32 bits drop such groups."""
    rows = ref.report_groups(80, mx, m) + ref.report_groups(81, mx, m) + ref.edge_rows(82, mx, n_random=100)
    full = ref.union([rows])
    rows = ref.rows_of(full)
    own, other = rows[0::2], rows[1::2] + rows[0::6]   # the list repeats some of the context's keys
    with api.DeviceContext(api.MODE_SHORT, mn, mx) as ctx:
        d = on_device(ref.to_array(own))
        ctx.merge_rows(d.data_ptr(), d.shape[0])
        ctx.set_report_filter(m)
        want_own = ref.filter_rule(ref.union([own]), m)
        check(finish_rows(ctx), ref.sorted_rows(want_own), "finish under the filter")
        dl = on_device(ref.to_array(other))
        want = ref.filter_rule(ref.union([own, other]), m)
        assert 0 < len(want) < len(full) or m == 1
        check(merged_rows(ctx, [(dl.data_ptr(), dl.shape[0])]), ref.sorted_rows(want), "union under the filter")
        ctx.set_report_filter(0)
        check(finish_rows(ctx), ref.sorted_rows(ref.union([own])), "filter off")


# ---- scan tables at scale against the oracle --------------------------------------------------------------------------
#
# Tables are linear in the reads and a unit (a read, a pair) leaves nothing behind for the next, so a batch built from a
# pool of units with multiplicities has the tables sum(multiplicity * tables of the unit alone); the oracle only scans
# the pool.  Shuffled batches of tens of thousands of distinct keys send far more than 256 distinct keys to each block
# (the thread kernels' staging table overflows into direct adds) while the hot units' keys are added from every block.

def units_64(seed, count):
    """150-base reads of one 33- to 64-base unit repeated, some with substitutions or a random flank."""
    import random
    rng = random.Random(seed)
    out = []
    for i in range(count):
        L = rng.randint(33, 64)
        unit = bytes(rng.choice(b"ACGT") for _ in range(L))
        ph = rng.randrange(L)
        r = bytearray((unit * (300 // L + 2))[ph:ph + 150])
        if i % 3 == 1:
            for _ in range(rng.randint(1, 4)):
                r[rng.randrange(150)] = rng.choice(b"ACGT")
        if i % 5 == 2:
            f = rng.randint(10, 60)
            r[:f] = bytes(rng.choice(b"ACGT") for _ in range(f))
        out.append(bytes(r))
    return out + synth.adversarial_short(seed + 1, count // 2, max_unit=64)


def multiplicities(seed, n_units, hot, hot_copies, tables):
    """Most units 1-3 copies; `hot` units with a non-empty table `hot_copies` copies each."""
    rng = np.random.default_rng(seed)
    mult = rng.integers(1, 4, n_units)
    productive = [i for i, t in enumerate(tables) if t]
    for i in rng.choice(productive, hot, replace=False):
        mult[i] = hot_copies
    return mult


def expected_tables(tables, mult):
    out = {}
    for t, m in zip(tables, mult.tolist()):
        for key, c in t.items():
            out[key] = out.get(key, 0) + m * c
    return out


def shuffled_batch(seed, mult):
    order = np.repeat(np.arange(len(mult)), mult)
    return order[np.random.default_rng(seed).permutation(order.size)]


SCALE = {   # name: (mode, min_mer, max_mer, slice, pool, hot units, copies of a hot unit)
    "short_5_32": (api.MODE_SHORT, 5, 32, 150, lambda: synth.adversarial_short(90, 8000), 20, 100_000),
    "short_3_64": (api.MODE_SHORT, 3, 64, 150, lambda: units_64(91, 4000), 20, 100_000),
    "paired_5_32": (api.MODE_PAIR, 5, 32, 150, lambda: synth.adversarial_pairs(92, 4000, read_len=150, max_unit=32), 10, 100_000),
    "long_5_32": (api.MODE_LONG, 5, 32, 150, lambda: synth.adversarial_long(93, 300, min_len=2000, max_len=5000, max_unit=32), 8, 4000),
}


@pytest.mark.parametrize("name", list(SCALE))
def test_scan_tables_at_scale(name):
    """Short 5 32 (64-bit keys through the staging table), short 3 64 with 33- to 64-base units (128-bit keys, added
    directly), paired 5 32 (the pair thread kernel) and long 5 32 at SLICE 150 on 2-5 kb reads (the warp kernel's direct
    adds): 2-4 M reads (30 k long reads) against the oracle's per-unit tables times their multiplicities."""
    from oracle.oracle import Oracle
    mode, mn, mx, sl, make_pool, hot, copies = SCALE[name]
    pool = make_pool()
    o = Oracle(mn, mx, slice_len=sl)
    if mode == api.MODE_PAIR:
        r1, r2 = pool
        units = list(dict.fromkeys(zip(r1, r2)))
        tables = [o.scan(1, [a], [b]) for a, b in units]
    else:
        units = list(dict.fromkeys(pool))
        tables = [o.scan(mode, [u]) for u in units]
    mult = multiplicities(100 + list(SCALE).index(name), len(units), hot, copies, tables)
    order = shuffled_batch(7, mult)
    want = expected_tables(tables, mult)
    with api.DeviceContext(mode, mn, mx, slice_length=sl) as ctx:
        if mode == api.MODE_PAIR:
            b1, l1 = api.make_chunk([units[i][0] for i in order])
            b2, l2 = api.make_chunk([units[i][1] for i in order])
            ctx.submit_chunk(b1, l1, b2, l2)
        else:
            b1, l1 = api.make_chunk([units[i] for i in order])
            ctx.submit_chunk(b1, l1)
        got = ctx.finish()
    assert len(want) > 1000 and max(want.values()) >= copies
    if mode != api.MODE_LONG:
        assert order.size >= 1_000_000
    assert got == want, "%d vs %d entries, first differences %s" % (len(got), len(want), sorted(set(got.items()) ^ set(want.items()))[:6])


def test_counts_past_2_32():
    """One resident short-mode batch of 2 M reads, half of them one telomeric read, scanned R times: its O_h / O_l
    TTAGGG rows pass 2^32.  finish(), finish() under set_report_filter(10) and the count the report prints equal R times
    the oracle's tables of the batch."""
    from oracle.oracle import Oracle, str_to_seq
    o = Oracle(5, 32)
    tel = b"TTAGGG" * 25
    units = [tel] + list(dict.fromkeys(synth.adversarial_short(95, 2000)))
    tables = [o.scan(0, [u]) for u in units]
    rng = np.random.default_rng(96)
    mult = rng.integers(250, 750, len(units))
    mult[0] = 1_000_000
    per_scan = expected_tables(tables, mult)
    hot = (4, 6, str_to_seq("TTAGGG"))
    R = (1 << 32) // per_scan[hot] + 2
    want = {key: R * c for key, c in per_scan.items()}
    assert want[hot] > 1 << 32
    order = shuffled_batch(97, mult)
    assert order.size > 1_900_000
    buf, locs = api.make_chunk([units[i] for i in order])
    pb = api.PackedBatch(buf, locs)
    pb.batch.max_read_len = max(len(u) for u in units)
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as ctx:
        h = ctx.upload(pb)
        for _ in range(R):
            ctx.scan_resident(h)
        got = ctx.finish()
        ctx.set_report_filter(10)
        kept = ctx.finish()
        ctx.free_resident(h)
    assert got == want, "%d vs %d entries" % (len(got), len(want))
    assert kept == ref.filter_rule(want, 10)
    texts = []
    for tables in (kept, want):
        rep = api.Report(5)
        rep.add_file("F", tables)
        texts.append(rep.finish())
    assert texts[0] == texts[1]
    assert ",%d," % want[hot] in texts[0] or ",%d\n" % want[hot] in texts[0]
