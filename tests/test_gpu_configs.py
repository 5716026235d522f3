"""The CUDA scan across the configuration grid (oracle/configs.py): k-mer bounds at the key and word boundaries, low and
extreme baselines, short slices.  Per configuration the tables equal the oracle's bit for bit; a subset runs with every
survivor on the warp kernel; unit records on one configuration per mode; the dense regime (LOW <= 0.2 on uniform random
reads: dozens of count-1 keys per read) at scale, on the default table and streamed through a small one that has to grow;
an overflow on a tiny table; and the `trew` binary with valid non-default -L / -H / -s values."""
import os
import random
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import configs as cf   # noqa: E402
from oracle.oracle import Oracle   # noqa: E402
from oracle_records import scan_records   # noqa: E402
from trew_b200 import api, synth   # noqa: E402

pytestmark = pytest.mark.gpu

NAMES = list(cf.CONFIGS)
STAGING = 1 << 18    # small staging slots: cheap contexts, several batches per configuration
TABLE_FULL = 3       # TREW_ERR_TABLE_FULL


def diff_msg(got, want):
    d = sorted(set(got.items()) ^ set(want.items()))
    return "%d vs %d entries, first differences %s" % (len(got), len(want), d[:6])


def context(name, **kw):
    mode, mn, mx, low, high, sl = cf.CONFIGS[name]
    kw.setdefault("staging_bytes", STAGING)
    return api.DeviceContext(mode, mn, mx, low, high, sl, **kw)


def scan(name, units, parts=3, **kw):
    """the units submitted in `parts` submissions to one context"""
    with context(name, **kw) as ctx:
        step = max(1, -(-len(units) // parts))
        for i in range(0, len(units), step):
            _, r1, r2 = cf.scan_args(name, units[i:i + step])
            ctx.submit_reads(r1, r2)
        return ctx.finish()


def differing_units(name, units):
    """the regimes and branch tags of the units whose records differ from the oracle's"""
    mode, r1, r2 = cf.scan_args(name, units)
    with context(name) as ctx:
        ctx.enable_unit_records(1 << 24)
        ctx.submit_reads(r1, r2)
        got = api.unit_records_dict(ctx.unit_records())
    exp = scan_records(cf.oracle_for(cf.CONFIGS[name]), mode, r1, r2)
    bad = sorted({unit for (unit, _, _, _), _ in set(got.items()) ^ set(exp.items())})
    return [(i, sorted(units[i].regimes)) for i in bad[:8]], len(bad)


def check(name, units, got, want):
    if got != want:
        pytest.fail("%s: %s; differing units %s" % (name, diff_msg(got, want), differing_units(name, units)))


@pytest.fixture(scope="module")
def corpora():
    t = time.time()
    c = {name: cf.corpus(name) for name in NAMES}
    w = {}
    for name in NAMES:
        mode, r1, r2 = cf.scan_args(name, c[name])
        w[name] = cf.oracle_for(cf.CONFIGS[name]).scan(mode, r1, r2)
    print("\nconfiguration corpora: %d configurations, %d units, generated and scanned by the oracle in %.1f s"
          % (len(NAMES), sum(map(len, c.values())), time.time() - t))
    return c, w


def test_tables_per_configuration(corpora):
    c, w = corpora
    for name in NAMES:
        check(name, c[name], scan(name, c[name]), w[name])
        assert w[name], name


# a subset spanning the table of boundaries: k 16 / 17, 31 / 32 / 33, MAX 37 / 38 / 40 / 41 / 63 / 64, the MIN_MER guards,
# the baselines, every mode and short slices
WARP_SUBSET = ("short_3_17", "short_19_33", "short_38_38", "short_40_41", "short_3_64", "pair_31_32", "pair_64_64",
               "long_3_64_s128", "long_5_23_s47", "short_5_32_1_1", "pair_5_32_0.050000000000000003_0.10000000000000001",
               "pair_5_32_0.33333333333333331_0.66666666666666663", "random_05")


def test_warp_kernel_for_every_survivor(corpora, monkeypatch):
    """TREW_EXACT_FLAGS=4: the thread kernel takes nothing; the warp kernel decides every survivor"""
    c, w = corpora
    monkeypatch.setenv("TREW_EXACT_FLAGS", "4")
    for name in WARP_SUBSET:
        got = scan(name, c[name])
        assert got == w[name], "%s (warp only): %s" % (name, diff_msg(got, w[name]))


RECORD_SUBSET = ("short_3_64", "pair_16_17", "long_3_32_s64", "short_5_32_0.10000000000000001_0.20000000000000001")


def test_unit_records(corpora):
    c, w = corpora
    for name in RECORD_SUBSET:
        mode, r1, r2 = cf.scan_args(name, c[name])
        with context(name) as ctx:
            ctx.enable_unit_records(1 << 24)
            ctx.submit_reads(r1, r2)
            got = api.unit_records_dict(ctx.unit_records())
            tables = ctx.finish()
        exp = scan_records(cf.oracle_for(cf.CONFIGS[name]), mode, r1, r2)
        assert got == exp, name + ": " + diff_msg(got, exp)
        summed = {}
        for (_, tb, k, s), n in got.items():
            summed[(tb, k, s)] = summed.get((tb, k, s), 0) + n
        assert summed == tables == w[name], name


# ---- the dense regime at scale ---------------------------------------------------------------------------------------------

# (mode, MIN, MAX, LOW, HIGH, units): about 32 distinct keys per 150-base read, 90 to 130 per pair (oracle), so that the
# rows stay below half of the default table (2^22 slots)
DENSE = [(0, 5, 32, 0.1, 0.2, 60000), (0, 3, 64, 0.05, 0.1, 60000), (1, 5, 32, 0.1, 0.2, 20000), (1, 3, 64, 0.05, 0.1, 15000)]


ACGT = bytes(b"ACGT"[i & 3] for i in range(256))


def uniform(seed, n, length=150):
    """n uniform random reads"""
    b = random.Random(seed).randbytes(n * length).translate(ACGT)
    return [b[i:i + length] for i in range(0, n * length, length)]


@pytest.mark.parametrize("mode,mn,mx,low,high,units", DENSE)
def test_dense_regime_at_scale(mode, mn, mx, low, high, units):
    r1 = uniform(1000 + mn + mx, units)
    r2 = uniform(2000 + mn + mx, units) if mode == 1 else None
    recs = scan_records(Oracle(mn, mx, low, high), mode, r1, r2)
    want, emitting = {}, set()
    for (u, tb, k, s), n in recs.items():
        want[(tb, k, s)] = want.get((tb, k, s), 0) + n
        emitting.add(u)
    assert (1 << 18) < len(want) < (1 << 21), len(want)   # grows a 2^20 table; below half of the default one
    # one batch on the default table
    with api.DeviceContext(mode, mn, mx, low, high) as ctx:
        ctx.submit_reads(r1, r2)
        got = ctx.finish()
        st = ctx.stats()
    assert got == want, diff_msg(got, want)
    assert st.survivors >= len(emitting) and len(emitting) > units // 4, (st.survivors, len(emitting))
    # streamed through small staging slots into a 2^20-slot table that has to grow between batches; each batch brings
    # fewer new keys than a quarter of the table
    staging = (1 << 18) if mode == 0 else (1 << 17)
    with api.DeviceContext(mode, mn, mx, low, high, table_log2_slots=20, staging_bytes=staging) as ctx:
        for i in range(0, units, 5000):
            ctx.submit_reads(r1[i:i + 5000], r2[i:i + 5000] if r2 else None)
        got = ctx.finish()
        st = ctx.stats()
    assert got == want, "streamed: " + diff_msg(got, want)
    assert st.units == units and st.survivors >= len(emitting)


def test_overflow_on_a_tiny_table():
    """one dense batch on a 2^10-slot table fails with TREW_ERR_TABLE_FULL instead of returning partial tables; after a
    reset, with the table grown, the same batch gives the oracle's tables"""
    reads = uniform(77, 2000)
    want = Oracle(5, 32, 0.1, 0.2).scan(0, reads)
    assert len(want) > 16 * (1 << 10)
    with api.DeviceContext(api.MODE_SHORT, 5, 32, 0.1, 0.2, table_log2_slots=10) as ctx:
        with pytest.raises(api.TrewError) as e:
            ctx.submit_reads(reads)
            ctx.finish()
        assert e.value.status == TABLE_FULL
        ctx.reset()
        ctx.reserve(len(want))
        ctx.submit_reads(reads)
        got = ctx.finish()
    assert got == want, diff_msg(got, want)


# ---- the command line with valid non-default values ------------------------------------------------------------------------

def report(min_mer, name, tables):
    r = api.Report(min_mer)
    r.add_file(name, tables)
    return r.finish()


def cli(args):
    return subprocess.run([api.CLI_PATH] + args, capture_output=True, check=True).stdout.decode()


def fastq(path, reads):
    with open(path, "wb") as f:
        f.write(synth.fastq_bytes(reads))
    return path


@pytest.mark.parametrize("mn,mx,low,high,spelling", [(5, 32, 0.1, 0.2, "short"), (3, 64, 0.35, 0.9, "short"),
                                                     (12, 40, 0.7, 0.7, "long_option")])
def test_cli_short_baselines(tmp_path, mn, mx, low, high, spelling):
    reads = synth.adversarial_short(300 + mn, 3000, max_unit=mx, lengths=[100, 150, 151]) + uniform(301, 500)
    p = fastq(str(tmp_path / "a.fastq"), reads)
    opts = ["-L", repr(low), "-H", repr(high)] if spelling == "short" else ["--low_baseline=%r" % low, "--high_baseline=%r" % high]
    out = cli(["short", str(mn), str(mx), p] + opts)
    exp = report(mn, os.path.realpath(p), Oracle(mn, mx, low, high).scan(0, reads))
    assert out == exp


def test_cli_paired_baselines(tmp_path):
    r1, r2 = synth.adversarial_pairs(310, 2000, read_len=150, max_unit=32, truncate_mate2=0.05)
    p1, p2 = fastq(str(tmp_path / "r_1.fastq"), r1), fastq(str(tmp_path / "r_2.fastq"), r2)
    out = cli(["short", "5", "32", "--paired_end", "--fq1", p1, "--fq2", p2, "-L", "0.3", "-H", "0.6"])
    exp = report(5, os.path.realpath(p1), Oracle(5, 32, 0.3, 0.6).scan(1, r1, r2))
    assert out == exp


@pytest.mark.parametrize("mn,mx,sl", [(3, 5, 10), (5, 23, 47)])
def test_cli_long_slices(tmp_path, mn, mx, sl):
    reads = synth.adversarial_long(320 + sl, 60, min_len=sl, max_len=3000, max_unit=mx)
    p = fastq(str(tmp_path / "l.fastq"), reads)
    out = cli(["long", str(mn), str(mx), p, "-s", str(sl), "-L", "0.4"])
    exp = report(mn, os.path.realpath(p), Oracle(mn, mx, 0.4, 0.8, slice_len=sl).scan(2, reads))
    assert out == exp
