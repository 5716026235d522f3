"""Per-unit hit records, checked without a GPU.  The oracle's per-unit records (each unit scanned alone,
tests/oracle_records.py) must sum to its tables of the whole input in every mode -- no unit leaves state behind for the
next, which is what makes them the records -- and the host build of the thread-per-read exact routing with a recording
emission (tests/native/unit_records_check.cpp) must give the oracle's records unit by unit, clean and under ASan + UBSan."""
import ctypes as C
import os
import subprocess
import sys
from collections import defaultdict

import numpy as np
import pytest

from oracle import edges
from oracle.oracle import Oracle
from trew_b200 import api, synth

from oracle_records import scan_records
from test_exact_thread import thr_table

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "native", "unit_records_check.cpp")


def summed(recs):
    """{(unit, table, k, seq): count} -> {(table, k, seq): count}"""
    out = defaultdict(int)
    for (_, tb, k, s), c in recs.items():
        out[(tb, k, s)] += c
    return dict(out)


def check_identity(o, mode, r1, r2=None):
    recs = scan_records(o, mode, r1, r2)
    assert summed(recs) == o.scan(mode, r1, r2)
    assert all(c > 0 for c in recs.values())
    assert all(0 <= u < len(r1) for (u, _, _, _) in recs)
    return recs


def test_oracle_records_sum_to_golden_tables(scan_cases):
    from test_oracle import tables_from_json
    for case in scan_cases:
        o = Oracle(case["min_mer"], case["max_mer"], case["low"], case["high"], case["slice_len"])
        r1 = [s.encode() for s in case["reads1"]]
        r2 = [s.encode() for s in case["reads2"]] if case["reads2"] is not None else None
        recs = scan_records(o, case["mode"], r1, r2)
        assert summed(recs) == tables_from_json(case["tables"]), case["name"]


@pytest.mark.parametrize("name", sorted(edges.CONFIGS))
def test_oracle_records_sum_to_tables_on_edges(name):
    mode, mn, mx, low, high, sl = edges.CONFIGS[name]
    _, r1, r2 = edges.scan_args(name, edges.corpus(name))
    recs = check_identity(Oracle(mn, mx, low, high, slice_len=sl), mode, r1, r2)
    assert len(recs) > 20


@pytest.mark.parametrize("mn,mx", [(5, 32), (3, 64), (12, 40)])
def test_oracle_records_sum_to_tables_adversarial(mn, mx):
    o = Oracle(mn, mx)
    # N runs (synth decorates reads with them), reads below 4 * MAX_MER and below 4 * MIN_MER, empty and all-N reads
    reads = synth.adversarial_short(31 + mx, 800, max_unit=mx, lengths=[150, 100, 60, 4 * mx - 1, 4 * mn - 1, 2 * mn])
    reads += [b"", b"N" * 150, b"TTAGGG" * 25, b"TTAGGGN" * 20]
    recs = check_identity(o, 0, reads)
    assert len({u for (u, _, _, _) in recs}) > 50
    r1, r2 = synth.adversarial_pairs(41 + mx, 500, read_len=150, max_unit=mx, truncate_mate2=0.2)   # truncated mates
    check_identity(o, 1, r1, r2)
    r1, r2 = synth.adversarial_pairs(43 + mx, 300, read_len=4 * mx - 3, max_unit=mx)   # pairs below 4 * MAX_MER
    check_identity(o, 1, r1, r2)


@pytest.mark.parametrize("sl", [150, 128])
def test_oracle_records_sum_to_tables_long(sl):
    o = Oracle(5, 32, slice_len=sl)
    # telomeric ends of a few hundred bases: the walks stop in the middle of the read
    reads = synth.adversarial_long(7 + sl, 120, min_len=sl - 20, max_len=3000)
    reads += [b"TTAGGG" * 80 + synth.adversarial_short(sl, 1, lengths=[900])[0], b"A" * (sl - 1)]
    recs = check_identity(o, 2, reads)
    assert any(tb in (2, 3) for (_, tb, _, _) in recs) and any(tb in (0, 1) for (_, tb, _, _) in recs)


# ---- the host build of the thread routing with a recording emission -------------------------------------------------------

def load(so):
    lib = C.CDLL(so)
    lib.urc_scan.restype = C.c_long
    lib.urc_scan.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                             C.c_void_p, C.c_void_p] + [C.c_void_p] * 6 + [C.c_long, C.POINTER(C.c_long), C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def urc(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("urc") / "liburc.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so, SRC])
    return load(so)


def run_records(lib, mode, r1, r2, mn, mx, sl=150, low=0.5, high=0.8):
    """(records {(unit, table, k, seq): count}, bailed unit indices) of the host thread routing"""
    b1, l1 = api.make_chunk(r1)
    l1 = np.ascontiguousarray(l1, dtype=np.int32)
    b2, l2 = api.make_chunk(r2) if r2 is not None else (np.zeros(1, np.uint8), np.zeros((1, 2), np.int32))
    l2 = np.ascontiguousarray(l2, dtype=np.int32)
    tl, th = thr_table(low), thr_table(high)
    cap = 1 << 20
    un, tb, kk = np.zeros(cap, np.uint64), np.zeros(cap, np.int32), np.zeros(cap, np.int32)
    lo, hi, ct = np.zeros(cap, np.uint64), np.zeros(cap, np.uint64), np.zeros(cap, np.uint64)
    nb = C.c_long(0)
    bi = np.zeros(max(1, len(r1)), np.int32)
    n = lib.urc_scan(mode, int(mx > 32), b1.tobytes(), l1.ctypes.data, b2.tobytes(), l2.ctypes.data, len(r1), mn, mx, sl, tl.ctypes.data,
                     th.ctypes.data, un.ctypes.data, tb.ctypes.data, kk.ctypes.data, lo.ctypes.data, hi.ctypes.data, ct.ctypes.data, cap,
                     C.byref(nb), bi.ctypes.data)
    assert n >= 0
    recs = {(int(un[i]), int(tb[i]), int(kk[i]), (int(hi[i]) << 64) | int(lo[i])): int(ct[i]) for i in range(n)}
    return recs, [int(x) for x in bi[:nb.value]]


def compare(lib, mode, r1, r2, mn, mx, sl=150, min_units=20):
    got, bailed = run_records(lib, mode, r1, r2, mn, mx, sl)
    skip = set(bailed)
    want = {key: c for key, c in scan_records(Oracle(mn, mx, slice_len=sl), mode, r1, r2).items() if key[0] not in skip}
    assert got == want, (len(got), len(want), sorted(set(got.items()) ^ set(want.items()))[:6])
    assert len({u for (u, _, _, _) in got}) >= min_units
    return bailed


@pytest.mark.parametrize("mn,mx", [(5, 32), (3, 64), (5, 40), (12, 64)])
def test_thread_records_equal_oracle_singles(urc, mn, mx):
    reads = synth.adversarial_short(2100 + mn * 7 + mx, 1500, max_unit=mx, lengths=[150, 160, 161, 128, 4 * mx - 1, 100, 60])
    bailed = compare(urc, 0, reads, None, mn, mx)
    assert bailed == [i for i, r in enumerate(reads) if len(r) > 160]   # reads that bail (the warp kernel's) record nothing here
    assert bailed


@pytest.mark.parametrize("mn,mx", [(5, 32), (3, 64), (5, 40), (12, 64)])
def test_thread_records_equal_oracle_pairs(urc, mn, mx):
    """At MAX_MER 64 every pair is below 4 * MAX_MER: all of them bail to the warp kernel and nothing is recorded here."""
    r1, r2 = synth.adversarial_pairs(2300 + mn * 7 + mx, 1200, read_len=160, max_unit=mx, truncate_mate2=0.15)
    bailed = compare(urc, 1, r1, r2, mn, mx, min_units=20 if 4 * mx <= 160 else 0)
    expect = [i for i, (a, b) in enumerate(zip(r1, r2))
              if min(len(a), len(b)) >= 2 * mn and (max(len(a), len(b)) > 160 or min(len(a), len(b)) < 4 * mx)]
    assert bailed == expect and bailed


@pytest.mark.parametrize("sl", [150, 128])
def test_thread_records_equal_oracle_long(urc, sl):
    from test_gpu_parity import config4_reads
    reads = synth.adversarial_long(2500 + sl, 150, min_len=sl - 10, max_len=4000) + config4_reads(sl, 48)
    bailed = compare(urc, 2, reads, None, 5, 32, sl)
    assert 0 < len(bailed) < len(reads) / 2


def test_thread_records_under_sanitizers(tmp_path):
    """The same harness in a library built with -fsanitize=address,undefined (workspace indices, shifts, record keys)."""
    so = os.path.join(str(tmp_path), "liburc_asan.so")
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                           "-Wno-unknown-pragmas", "-o", so, SRC])
    asan = subprocess.check_output(["g++", "-print-file-name=libasan.so"]).decode().strip()
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "native", "unit_records_sanitize.py"), so], env=env,
                       capture_output=True, timeout=900)
    assert r.returncode == 0 and b"sanitizer run clean" in r.stdout, (r.stdout[-500:], r.stderr[-3000:])
