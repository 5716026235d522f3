#!/usr/bin/env python3
"""Hit rate of classify_runs' rotation memo (exact_thread.cuh, kMemo entries), counted on the host build of the thread
path: every probe of the reads below goes through route_short_thread at MIN_MER 5, MAX_MER 32.

    python tools/memo_hits.py [reads]
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_exact_thread as t  # noqa: E402
from trew_b200 import synth  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 200_000
with tempfile.TemporaryDirectory() as d:
    so = os.path.join(d, "libmemo.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so,
                           os.path.join(ROOT, "tools", "memo_hits.cpp")])
    lib = C.CDLL(so)
lib.etc_scan_reads.restype = C.c_long
lib.etc_scan_reads.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_long, C.POINTER(C.c_long), C.c_void_p]
lib.etc_memo_runs.restype = C.c_long
lib.etc_memo_hits.restype = C.c_long
sets = [("bench shape (configs[1])", synth.config_short(3, n)),
        ("telomeric reads only", synth.config_short(4, max(1, n // 10), telomeric=1.0, half_telomeric=0.0))]
for name, rows in sets:
    lib.etc_memo_reset()
    t.run(lib, [bytes(r) for r in rows], 5, 32)
    r, h = lib.etc_memo_runs(), lib.etc_memo_hits()
    print("%-26s %8d reads  exact-mode runs %9d  memo hits %9d  = %.1f %%" % (name, len(rows), r, h, 100.0 * h / max(1, r)))
