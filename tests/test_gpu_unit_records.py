"""Per-unit hit records on the GPU: the device's records equal the oracle's unit by unit (both exact kernels, the long
three-step path and the warp kernel's bail list), sum to the tables of finish() on bench-shaped batches, leave the tables
as they are, number units across chunks, batches, packed submissions and the devices of a group, and report an overflow
with the capacity that is enough.

Run as a script (what the TREW_EXACT_FLAGS test does in a child process), this file prints the device records of every
case of CASES as JSON."""
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle_records import scan_records   # noqa: E402
from trew_b200 import api, synth   # noqa: E402

pytestmark = pytest.mark.gpu

CAP = 1 << 22


def device_records(mode, mn, mx, low, high, sl, r1, r2=None, **kw):
    with api.DeviceContext(mode, mn, mx, low, high, sl, **kw) as ctx:
        ctx.enable_unit_records(CAP)
        ctx.submit_reads(r1, r2)
        recs = api.unit_records_dict(ctx.unit_records())
        return recs, ctx.finish()


def summed(recs):
    out = {}
    for (_, tb, k, s), c in recs.items():
        out[(tb, k, s)] = out.get((tb, k, s), 0) + c
    return out


def diff_msg(got, want):
    d = sorted(set(got.items()) ^ set(want.items()))
    return "%d vs %d records, first differences %s" % (len(got), len(want), d[:6])


def cases():
    """(name, mode, mn, mx, low, high, sl, reads1, reads2): both exact kernels (reads of up to 160 bases go to the thread
    kernel, longer ones and the rest to the warp kernel), short reads and pairs below 4 * MAX_MER, truncated mates, long
    reads whose walks stop inside the read"""
    out = []
    for mn, mx, low, high in [(5, 32, 0.5, 0.8), (3, 64, 0.5, 0.8), (7, 20, 0.5, 0.8), (12, 40, 0.5, 0.8), (5, 32, 0.35, 0.6), (5, 32, 0.9, 1.0)]:
        reads = synth.adversarial_short(3100 + mn * 7 + mx, 900, max_unit=mx, lengths=[150, 160, 161, 250, 100, 4 * mx - 1, 60])
        out.append(("short_%d_%d_%g_%g" % (mn, mx, low, high), 0, mn, mx, low, high, 150, reads, None))
    for mn, mx, rl in [(5, 32, 150), (3, 64, 150), (7, 20, 100), (12, 40, 200), (5, 32, 100)]:
        r1, r2 = synth.adversarial_pairs(3300 + mn * 7 + mx + rl, 600, read_len=rl, max_unit=mx, truncate_mate2=0.15)
        out.append(("pair_%d_%d_%d" % (mn, mx, rl), 1, mn, mx, 0.5, 0.8, 150, r1, r2))
    from test_gpu_parity import config4_reads
    for sl, mx in [(150, 32), (128, 32), (150, 64)]:
        reads = synth.adversarial_long(3500 + sl + mx, 120, min_len=sl - 10, max_len=4000, max_unit=mx) + config4_reads(sl + mx, 24)
        out.append(("long_%d_%d" % (sl, mx), 2, 5, mx, 0.5, 0.8, sl, reads, None))
    return out


def oracle_records(case):
    from oracle.oracle import Oracle
    name, mode, mn, mx, low, high, sl, r1, r2 = case
    return scan_records(Oracle(mn, mx, low, high, slice_len=sl), mode, r1, r2)


@pytest.fixture(scope="module")
def all_cases():
    cs = cases()
    return cs, {c[0]: oracle_records(c) for c in cs}


def test_records_equal_oracle(all_cases):
    cs, want = all_cases
    for c in cs:
        name, mode, mn, mx, low, high, sl, r1, r2 = c
        got, tables = device_records(mode, mn, mx, low, high, sl, r1, r2)
        assert got == want[name], name + ": " + diff_msg(got, want[name])
        assert summed(got) == tables, name
        assert all(v > 0 for v in got.values()) and len(got) > 50, name


@pytest.mark.parametrize("name", sorted(__import__("oracle.edges", fromlist=["CONFIGS"]).CONFIGS))
def test_records_equal_oracle_on_edges(name):
    from oracle import edges
    from oracle.oracle import Oracle
    mode, mn, mx, low, high, sl = edges.CONFIGS[name]
    _, r1, r2 = edges.scan_args(name, edges.corpus(name))
    got, tables = device_records(mode, mn, mx, low, high, sl, r1, r2)
    want = scan_records(Oracle(mn, mx, low, high, slice_len=sl), mode, r1, r2)
    assert got == want, name + ": " + diff_msg(got, want)
    assert summed(got) == tables


def run_cases_json():
    out = {}
    for name, mode, mn, mx, low, high, sl, r1, r2 in cases():
        got, _ = device_records(mode, mn, mx, low, high, sl, r1, r2)
        out[name] = [[u, tb, k, str(s), c] for (u, tb, k, s), c in sorted(got.items())]
    return out


@pytest.mark.parametrize("flags", ["4", "1", "2", "16"])
def test_records_under_exact_flags(all_cases, flags):
    """4: no thread kernel (everything through the warp kernel); 1, 2: the warp kernel's serial / bound switches; 16: long reads
    through the three-step thread path"""
    cs, want = all_cases
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=dict(os.environ, TREW_EXACT_FLAGS=flags), capture_output=True,
                       timeout=1200)
    assert r.returncode == 0, r.stderr.decode()[-3000:]
    got = json.loads(r.stdout)
    for name in want:
        g = {(u, tb, k, int(s)): c for u, tb, k, s, c in got[name]}
        assert g == want[name], name + " flags " + flags + ": " + diff_msg(g, want[name])


# ---- bench-shaped batches synthesised on the device ----------------------------------------------------------------------

def sum_by_key(v, count="count"):
    """structured rows -> (meta, seq_hi, seq_lo) sorted unique keys and summed counts"""
    meta = v["table"].astype(np.uint64) << np.uint64(8) | v["k"].astype(np.uint64)
    order = np.lexsort((v["seq_lo"], v["seq_hi"], meta))
    m, h, lo, c = meta[order], v["seq_hi"][order], v["seq_lo"][order], v[count][order].astype(np.uint64)
    head = np.ones(len(m), dtype=bool)
    head[1:] = (m[1:] != m[:-1]) | (h[1:] != h[:-1]) | (lo[1:] != lo[:-1])
    idx = np.flatnonzero(head)
    return m[idx], h[idx], lo[idx], np.add.reduceat(c, idx) if len(c) else c


def synth_scan(flavor, n_reads, read_len, batches, mode, rec_cap):
    with api.DeviceContext(mode, 5, 32) as ctx:
        if rec_cap:
            ctx.enable_unit_records(rec_cap)
        hs = [ctx.synth_resident(1000 + 17 * i + flavor, n_reads, read_len, tel_ppm=20000, flavor=flavor) for i in range(batches)]
        for h in hs:
            ctx.scan_resident(h)
        recs = ctx.unit_records() if rec_cap else None
        tables = ctx.finish_view().copy()
        for h in hs:
            ctx.free_resident(h)
    return recs, tables


@pytest.mark.parametrize("flavor,n_reads,read_len,batches,mode", [(0, 2_000_000, 150, 3, api.MODE_SHORT), (1, 2_000_000, 150, 2, api.MODE_PAIR),
                                                                   (2, 40_000, 15000, 2, api.MODE_LONG)])
def test_identity_on_synthetic_batches(flavor, n_reads, read_len, batches, mode):
    recs, tables = synth_scan(flavor, n_reads, read_len, batches, mode, 1 << 27)
    _, plain = synth_scan(flavor, n_reads, read_len, batches, mode, 0)
    assert np.array_equal(tables, plain)   # records on: the same tables
    units = n_reads // 2 if mode == api.MODE_PAIR else n_reads
    assert len(recs) > 1000 and recs["count"].min() > 0 and recs["reserved"].max() == 0
    assert recs["unit"].max() < units * batches and recs["unit"].max() >= units * (batches - 1)   # ordinals continue across batches
    key = np.stack([recs["unit"], recs["table"].astype(np.uint64), recs["k"].astype(np.uint64), recs["seq_hi"], recs["seq_lo"]])
    assert (np.diff(np.lexsort(key[::-1])) > 0).all()   # already sorted by (unit, table, k, seq_hi, seq_lo) ...
    same = (np.diff(key, axis=1) == 0).all(axis=0)
    assert not same.any()   # ... one row per key
    m, h, lo, c = sum_by_key(recs)
    tm, th, tlo, tc = sum_by_key(tables)
    assert np.array_equal(m, tm) and np.array_equal(h, th) and np.array_equal(lo, tlo) and np.array_equal(c, tc)


# ---- ordinals -----------------------------------------------------------------------------------------------------------

def test_ordinals_across_chunks_batches_and_packed():
    from oracle.oracle import Oracle
    reads = synth.adversarial_short(41, 3000, lengths=[150, 100, 161, 60])
    parts = [reads[:700], reads[700:1500], reads[1500:2200], reads[2200:]]
    with api.DeviceContext(api.MODE_SHORT, 5, 32, staging_bytes=1 << 16) as ctx:   # small staging: several batches per chunk
        ctx.enable_unit_records(CAP)
        ctx.submit_reads(parts[0])
        ctx.submit_reads(parts[1])
        buf, locs = api.make_chunk(parts[2])
        ctx.submit_packed(api.PackedBatch(buf, locs))
        ctx.submit_reads(parts[3])
        got = api.unit_records_dict(ctx.unit_records())
        assert summed(got) == ctx.finish()
        ctx.reset()   # clears the records and restarts the ordinals
        ctx.submit_reads(parts[3])
        again = api.unit_records_dict(ctx.unit_records())
    want = scan_records(Oracle(5, 32), 0, reads)
    assert got == want, diff_msg(got, want)
    off = 2200
    assert again == {(u - off, tb, k, s): c for (u, tb, k, s), c in want.items() if u >= off}


def test_enable_only_on_an_empty_table():
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as ctx:
        ctx.submit_reads([b"TTAGGG" * 25])
        with pytest.raises(api.TrewError) as e:
            ctx.enable_unit_records(100)
        assert e.value.status == 1
        ctx.reset()
        ctx.enable_unit_records(100)
        ctx.submit_reads([b"TTAGGG" * 25])
        r = ctx.unit_records()
        assert len(r) > 0 and set(r["unit"].tolist()) == {0}   # the ordinals restarted


def test_multi_context_on_one_device_equals_one_context():
    reads = synth.adversarial_short(43, 4000, lengths=[150, 100, 161])
    r1, r2 = synth.adversarial_pairs(44, 1500, truncate_mate2=0.1)
    for mode, a, b in [(api.MODE_SHORT, reads, None), (api.MODE_PAIR, r1, r2)]:
        one, _ = device_records(mode, 5, 32, 0.5, 0.8, 150, a, b)
        with api.MultiContext(mode, 5, 32, devices=[0, 0, 0]) as m:
            m.enable_unit_records(CAP)
            m.submit_reads(a, b, chunk_reads=300)
            got = api.unit_records_dict(m.unit_records())
            assert summed(got) == m.finish()
            m.reset()
            m.submit_reads(a[:300], b[:300] if b else None, chunk_reads=100)
            again = api.unit_records_dict(m.unit_records())
        assert got == one, diff_msg(got, one)
        assert again == {key: c for key, c in one.items() if key[0] < 300}


@pytest.mark.parametrize("kind", ["plain", "gzip", "bgzf"])
def test_process_file_ordinals_are_file_records(tmp_path, kind):
    from oracle.oracle import Oracle
    reads = synth.adversarial_short(45, 2500, lengths=[150, 100, 161])
    r1, r2 = synth.adversarial_pairs(46, 1200, truncate_mate2=0.1)
    # long mode: reads shorter than SLICE_LENGTH interleaved (the reader drops them, they keep their file index)
    lr = synth.adversarial_long(48, 200, min_len=150, max_len=3000)
    lr = [x for i, r in enumerate(lr) for x in ((r, r[: 1 + 7 * i % 148]) if i % 3 == 0 else (r,))]
    assert sum(len(r) < 150 for r in lr) > 50
    for mode, a, b in [(api.MODE_SHORT, reads, None), (api.MODE_PAIR, r1, r2), (api.MODE_LONG, lr, None)]:
        paths = []
        for i, rs in enumerate([a, b] if b else [a]):
            plain = str(tmp_path / ("m%d_%d.fq" % (mode, i)))
            open(plain, "wb").write(synth.fastq_bytes(rs))
            if kind == "gzip":
                open(plain + ".gz", "wb").write(gzip.compress(open(plain, "rb").read()))
                plain += ".gz"
            elif kind == "bgzf":
                synth.bgzf_write(plain, plain + ".bgz")
                plain += ".bgz"
            paths.append(plain)
        with api.DeviceContext(mode, 5, 32) as ctx:
            ctx.enable_unit_records(CAP)
            ctx.process_file(*paths)
            got = api.unit_records_dict(ctx.unit_records())
            tables = ctx.finish()
        with api.DeviceContext(mode, 5, 32) as ctx:
            ctx.process_file(*paths)
            assert ctx.finish() == tables == summed(got)
        want = scan_records(Oracle(5, 32), mode, a, b)
        assert got == want, (mode, diff_msg(got, want))


def test_capacity_overflow_names_the_capacity_that_is_enough():
    import re
    reads = synth.adversarial_short(47, 3000, lengths=[150, 100])
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as ctx:
        ctx.enable_unit_records(1000)
        ctx.submit_reads(reads)
        with pytest.raises(api.TrewError) as e:
            ctx.unit_records()
        assert e.value.status == 3
        need = int(re.search(r"a capacity of (\d+) is enough", str(e.value)).group(1))
        assert need > 1000
        full_tables = ctx.finish()   # the tables are not affected
        ctx.reset()
        ctx.enable_unit_records(need)
        ctx.submit_reads(reads)
        recs = ctx.unit_records()
        assert summed(api.unit_records_dict(recs)) == full_tables == ctx.finish()
    want, _ = device_records(api.MODE_SHORT, 5, 32, 0.5, 0.8, 150, reads)
    assert full_tables == summed(want) and len(recs) <= need


# ---- trew --read_hits ------------------------------------------------------------------------------------------------------

def fastq_reads(path):
    data = (gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb")).read()
    return data.split(b"\n")[1::4][: data.count(b"\n") // 4]


def oracle_tsv(path, mode, r1, r2=None, mn=5, mx=32):
    from oracle.oracle import Oracle, seq_to_str
    recs = scan_records(Oracle(mn, mx), mode, r1, r2)
    return "".join("%s\t%d\t%s\t%d\t%s\t%d\n" % (os.path.realpath(path), u, api.TABLE_NAMES[tb], k, seq_to_str(s, k), c)
                   for (u, tb, k, s), c in sorted(recs.items()))


def cli(args, hits=None):
    r = subprocess.run([api.CLI_PATH] + args + (["--read_hits", hits] if hits else []), capture_output=True, timeout=600)
    return r.returncode, r.stdout


def test_cli_read_hits(tmp_path):
    fx = os.path.join(ROOT, "tests", "golden", "fixtures")
    runs = []
    for name, sub in [("test.fastq", "short"), ("test.fastq.gz", "short"), ("test_long.fastq", "long"), ("test_long.fastq.gz", "long")]:
        p = os.path.join(fx, name)
        runs.append(([sub, "5", "32", p], oracle_tsv(p, 0 if sub == "short" else 2, fastq_reads(p))))
    r1, r2 = synth.adversarial_pairs(49, 1500, truncate_mate2=0.1)
    p1, p2 = str(tmp_path / "p_1.fq"), str(tmp_path / "p_2.fq")
    open(p1, "wb").write(synth.fastq_bytes(r1))
    open(p2, "wb").write(synth.fastq_bytes(r2))
    runs.append((["short", "5", "32", "--paired_end", "--fq1", p1, "--fq2", p2], oracle_tsv(p1, 1, r1, r2)))
    # all-telomeric reads: more records than the capacity the input's size gives, so the file is scanned a second time
    tel = [bytes(r) for r in synth.config_short(50, 3000, telomeric=1.0, sub=0.03)]
    pt = str(tmp_path / "tel.fq")
    open(pt, "wb").write(synth.fastq_bytes(tel))
    want_tel = oracle_tsv(pt, 0, tel)
    assert want_tel.count("\n") > max(os.path.getsize(pt) // 128, 1 << 12)
    runs.append((["short", "5", "32", pt], want_tel))
    # two files in one run: each file's records, its own ordinals
    two = oracle_tsv(runs[0][0][3], 0, fastq_reads(runs[0][0][3])) + want_tel
    runs.append((["short", "5", "32", runs[0][0][3], pt], two))
    for args, want in runs:
        hits = str(tmp_path / "hits.tsv")
        rc0, out0 = cli(args)
        rc1, out1 = cli(args, hits)
        assert rc0 == rc1 == 0 and out0 == out1 and out0, args
        got = open(hits).read()
        assert got == want, (args, got.count("\n"), want.count("\n"))


if __name__ == "__main__":
    json.dump(run_cases_json(), sys.stdout)
