"""The CUDA scan on windows of 161 up to 1023 bases (oracle/long_windows.py), where only the warp-per-survivor exact kernel
decides: tables bit-exact with the oracle per configuration, per length and per constructed regime; batches that mix
lengths (a read's probe longer than the filter variant its batch's longest read picks, one long pair among short ones,
a second batch longer than the first); the routing switches; unit records; the length limits through every entry point;
and paired files of 2 x 250 and 2 x 300 bases."""
import ctypes as C
import os
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import long_windows as lw   # noqa: E402
from oracle.oracle import Oracle   # noqa: E402
from oracle_records import scan_records   # noqa: E402
from trew_b200 import api, synth   # noqa: E402

pytestmark = pytest.mark.gpu

NAMES = list(lw.CONFIGS)


def diff_msg(got, want):
    d = sorted(set(got.items()) ^ set(want.items()))
    return "%d vs %d entries, first differences %s" % (len(got), len(want), d[:6])


def oracle_for(name):
    mode, mn, mx, low, high, sl = lw.CONFIGS[name]
    return Oracle(mn, mx, low, high, slice_len=sl)


def context(name, **kw):
    mode, mn, mx, low, high, sl = lw.CONFIGS[name]
    return api.DeviceContext(mode, mn, mx, low, high, sl, **kw)


def scan(name, units, **kw):
    _, r1, r2 = lw.scan_args(name, units)
    with context(name, **kw) as ctx:
        ctx.submit_reads(r1, r2)
        return ctx.finish()


def want(name, units):
    mode, r1, r2 = lw.scan_args(name, units)
    return oracle_for(name).scan(mode, r1, r2)


@pytest.fixture(scope="module")
def corpora():
    t = time.time()
    c = {name: lw.corpus(name) for name in NAMES}
    w = {name: want(name, c[name]) for name in NAMES}
    print("\nlong-window corpora: %d units, generated and scanned by the oracle in %.1f s" % (sum(map(len, c.values())), time.time() - t))
    return c, w


def test_tables_per_configuration_and_length(corpora):
    c, w = corpora
    for name in NAMES:
        got = scan(name, c[name])
        assert got == w[name], name + ": " + diff_msg(got, w[name])
        assert len(w[name]) > 50, name
        # one length at a time, in one context reset between them, so that a failure names its length
        with context(name) as ctx:
            for key in lw.lengths(name):
                sub = [u for u in c[name] if u.length == key and not u.regimes & set(lw.REGIMES)]
                _, r1, r2 = lw.scan_args(name, sub)
                ctx.reset()
                ctx.submit_reads(r1, r2)
                got, exp = ctx.finish(), want(name, sub)
                assert got == exp, "%s length %s: %s" % (name, key, diff_msg(got, exp))


def test_tables_per_regime(corpora):
    c, _ = corpora
    seen = set()
    for name in NAMES:
        for regime in lw.REGIMES:
            sub = [u for u in c[name] if regime in u.regimes]
            if not sub:
                continue
            seen.add(regime)
            got, exp = scan(name, sub), want(name, sub)
            assert got == exp and exp, "%s %s: %s" % (name, regime, diff_msg(got, exp))
    assert seen == set(lw.REGIMES)


# ---- batches that mix lengths --------------------------------------------------------------------------------------------

def one_batch_and_per_length(name, groups, **kw):
    """tables of all groups in one submission, of each group in a submission of its own (one context), and the oracle's"""
    mode = lw.CONFIGS[name][0]
    mixed = [u for g in groups for u in g]
    rng = __import__("random").Random(len(mixed))
    rng.shuffle(mixed)
    one = scan(name, mixed, **kw)
    with context(name, **kw) as ctx:
        for g in groups:
            _, r1, r2 = lw.scan_args(name, g)
            ctx.submit_reads(r1, r2)
        split = ctx.finish()
    return one, split, want(name, mixed)


def units_of(reads1, reads2=None):
    return [lw.Unit([a] if reads2 is None else [a, b], len(a), ()) for a, b in zip(reads1, reads2 or reads1)]


@pytest.mark.parametrize("name,long_len,short_len", [("short_5_32", 190, 127), ("short_3_64", 300, 255), ("short_3_64", 1000, 255),
                                                     ("short_12_40", 999, 159)])
def test_mixed_lengths_probe_longer_than_the_batch_variant(name, long_len, short_len):
    """the filter variant comes from the longest read's half (95 bases at 190, 150 at 300); the shorter reads are below
    4 * MAX_MER and probe their whole read (127, 255 bases)"""
    mx = lw.CONFIGS[name][2]
    a = units_of(synth.adversarial_short(61 + long_len, 200, max_unit=mx, lengths=[long_len]))
    b = units_of(synth.adversarial_short(62 + short_len, 400, max_unit=mx, lengths=[short_len]))
    b += units_of([(b"TTAGGG" * 60)[:short_len], (b"ACG" * 90)[:short_len], (b"TTAGGC" * 60)[:short_len]])
    one, split, exp = one_batch_and_per_length(name, [a, b])
    assert one == exp, diff_msg(one, exp)
    assert split == exp, diff_msg(split, exp)


@pytest.mark.parametrize("name", ["pair_5_32", "pair_3_64"])
def test_one_long_pair_among_short_pairs(name):
    mx = lw.CONFIGS[name][2]
    r1, r2 = synth.adversarial_pairs(70 + mx, 1500, read_len=150, max_unit=mx, truncate_mate2=0.1)
    l1, l2 = synth.adversarial_pairs(71 + mx, 1, read_len=1023, max_unit=mx)
    long_pair = units_of([(b"TTAGGG" * 171)[:1023]], [(b"CCCTAA" * 171)[:1023]]) + units_of(l1, l2)
    one, split, exp = one_batch_and_per_length(name, [units_of(r1, r2), long_pair])
    assert one == exp, diff_msg(one, exp)
    assert split == exp, diff_msg(split, exp)


@pytest.mark.parametrize("name,first,second", [("short_5_32", 150, 1000), ("pair_3_64", 150, 1023), ("long_5_32_s64", 2000, 60000),
                                               ("long_5_32_s512", 600, 20000)])
def test_second_batch_longer_than_the_first(name, first, second):
    """the exact kernel's run capacity and the long-read scratch grow between batches; a small staging buffer splits each
    submission into several batches"""
    mode, mn, mx, _, _, sl = lw.CONFIGS[name]

    def reads(seed, n, count):
        if mode == 0:
            return units_of(synth.adversarial_short(seed, count, max_unit=mx, lengths=[n]))
        if mode == 1:
            return units_of(*synth.adversarial_pairs(seed, count, read_len=n, max_unit=mx))
        return units_of(synth.adversarial_long(seed, count, min_len=n // 2, max_len=n, max_unit=mx))
    a, b = reads(80 + first, first, 300), reads(81 + second, second, 40)
    with context(name, staging_bytes=1 << 16) as ctx:
        for g in (a, b, a):
            _, r1, r2 = lw.scan_args(name, g)
            ctx.submit_reads(r1, r2)
        got = ctx.finish()
        st = ctx.stats()
    exp = want(name, a + b + a)
    assert got == exp, diff_msg(got, exp)
    assert st.units == 2 * len(a) + len(b)


# ---- routing switches ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("flags", ["1", "2"])
def test_exact_flags(corpora, monkeypatch, flags):
    """1: eval_k's serial path for every evaluation; 2: without comp_bound"""
    c, w = corpora
    monkeypatch.setenv("TREW_EXACT_FLAGS", flags)
    for name in NAMES:
        got = scan(name, c[name])
        assert got == w[name], "%s flags %s: %s" % (name, flags, diff_msg(got, w[name]))


def test_long_three_kernel_path(corpora, monkeypatch):
    """TREW_EXACT_FLAGS=16: at SLICE 160 the three-kernel long path takes slices of up to 160 bases and the mid slices
    above 160 still go to the warp kernel; at SLICE 161 the path does not apply"""
    c, w = corpora
    monkeypatch.setenv("TREW_EXACT_FLAGS", "16")
    for name in ("long_5_32_s160", "long_3_64_s160", "long_5_32_s161", "long_3_64_s161", "long_5_32_s128", "long_5_32_s64"):
        got = scan(name, c[name])
        assert got == w[name], name + ": " + diff_msg(got, w[name])


# ---- unit records --------------------------------------------------------------------------------------------------------

def test_unit_records(corpora):
    c, _ = corpora
    picks = {
        "pair_5_32": lambda u: 1023 in (len(u.mates[0]), len(u.mates[1])),
        "pair_3_64": lambda u: 1023 in (len(u.mates[0]), len(u.mates[1])),
        "long_5_32_s512": lambda u: True,
        "long_3_64_s512": lambda u: True,
        "short_5_32": lambda u: len(u.mates[0]) >= 999,
        "short_3_64": lambda u: len(u.mates[0]) >= 999,
    }
    for name, pick in picks.items():
        sub = [u for u in c[name] if pick(u)]
        mode, r1, r2 = lw.scan_args(name, sub)
        with context(name) as ctx:
            ctx.enable_unit_records(1 << 22)
            ctx.submit_reads(r1, r2)
            got = api.unit_records_dict(ctx.unit_records())
        exp = scan_records(oracle_for(name), mode, r1, r2)
        assert len(sub) >= 8 and exp, name
        assert got == exp, name + ": " + diff_msg(got, exp)


# ---- length limits ---------------------------------------------------------------------------------------------------------

def status_of(fn):
    try:
        fn()
    except api.TrewError as e:
        return e.status
    return 0


def packed(reads1, reads2=None):
    buf, locs = api.make_chunk(reads1)
    if reads2 is None:
        return api.PackedBatch(buf, locs)
    buf2, locs2 = api.make_chunk(reads2)
    return api.PackedBatch(buf, locs, n_ranges=1, buf2=buf2, locs2=locs2)


def check_batch(mode, pb):
    return api.load_library().trew_check_batch(mode, C.byref(pb.batch))


@pytest.mark.parametrize("mode,ok,over", [(api.MODE_SHORT, 1000, 1001), (api.MODE_PAIR, 1023, 1024)])
def test_length_limits_through_every_entry_point(mode, ok, over):
    """submit_reads, submit_packed and upload: the longest accepted read scans like the oracle, one base more gives
    TREW_ERR_TOO_LONG before anything is launched"""
    tel = (b"TTAGGG" * 200)[:ok]
    r_ok = [tel, synth.adversarial_short(90, 1, lengths=[ok])[0]]
    r_over = [(b"TTAGGG" * 200)[:over]]
    pair = mode == api.MODE_PAIR
    exp = Oracle(5, 32).scan(mode, r_ok, r_ok if pair else None)
    with api.DeviceContext(mode, 5, 32) as ctx:
        ctx.submit_reads(r_ok, r_ok if pair else None)
        assert ctx.finish() == exp
        ctx.reset()
        pb = packed(r_ok, r_ok if pair else None)
        assert pb.batch.max_read_len == ok
        ctx.submit_packed(pb)
        assert ctx.finish() == exp
        ctx.reset()
        h = ctx.upload(pb)
        ctx.scan_resident(h)
        assert ctx.finish() == exp
        ctx.free_resident(h)
    with api.DeviceContext(mode, 5, 32) as ctx:
        assert status_of(lambda: ctx.submit_reads(r_over, r_over if pair else None)) == 4
        pb_over = packed(r_over, r_over if pair else None)
        assert check_batch(mode, pb_over) == 4
        assert status_of(lambda: ctx.submit_packed(pb_over)) == 4
        assert status_of(lambda: ctx.upload(pb_over)) == 4
        assert ctx.stats().units == 0 and ctx.finish() == {}   # nothing of the refused batches was scanned


def test_packed_max_read_len():
    """a larger max_read_len only sizes the workspace up; a smaller one is refused (checked on the host first)"""
    reads = synth.adversarial_short(91, 300, lengths=[1000, 700, 161, 150]) + [(b"ACG" * 400)[:1000]]
    exp = Oracle(5, 32).scan(0, reads)
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as ctx:
        pb = packed(reads)
        ctx.submit_packed(pb, max_read_len=1023)
        assert ctx.finish() == exp
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as ctx:
        pb = packed(reads)
        pb.batch.max_read_len = 999
        assert check_batch(api.MODE_SHORT, pb) == 1   # refused on the host: the scan below never starts
        assert status_of(lambda: ctx.submit_packed(pb)) == 1
        assert status_of(lambda: ctx.upload(pb)) == 1
        assert status_of(lambda: ctx.submit_packed(packed(reads), max_read_len=150)) == 1
        assert ctx.finish() == {}


def test_slice_length_limits():
    r = [(b"TTAGGG" * 400)[:2047], (b"ACG" * 400)[:1023]]
    with api.DeviceContext(api.MODE_LONG, 5, 32, slice_length=512) as ctx:
        ctx.submit_reads(r)
        assert ctx.finish() == Oracle(5, 32, slice_len=512).scan(2, r)
    for sl, mx in [(513, 32), (63, 32), (127, 64)]:
        with pytest.raises(api.TrewError) as e:
            api.DeviceContext(api.MODE_LONG, 5, mx, slice_length=sl)
        assert e.value.status == 1, (sl, mx)


# ---- files ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("read_len", [250, 300])
def test_paired_files(tmp_path, read_len):
    r1, r2 = synth.adversarial_pairs(95 + read_len, 1500, read_len=read_len, truncate_mate2=0.05)
    p1, p2 = str(tmp_path / "r_1.fq"), str(tmp_path / "r_2.fq")
    open(p1, "wb").write(synth.fastq_bytes(r1))
    open(p2, "wb").write(synth.fastq_bytes(r2))
    with api.DeviceContext(api.MODE_PAIR, 5, 32) as ctx:
        ctx.process_file(p1, p2)
        from_file = ctx.finish()
    with api.DeviceContext(api.MODE_PAIR, 5, 32) as ctx:
        ctx.submit_reads(r1, r2)
        from_reads = ctx.finish()
    exp = Oracle(5, 32).scan(1, r1, r2)
    assert from_file == from_reads == exp, diff_msg(from_file, exp)
