"""Driver of tests/test_unit_records.py::test_thread_records_under_sanitizers: the recording host build of the thread
routing (short, paired, long; 64- and 128-bit keys; reads that bail) inside a library compiled with
-fsanitize=address,undefined, each run diffed against the oracle.  usage: LD_PRELOAD=libasan.so python unit_records_sanitize.py liburc_asan.so"""
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_unit_records as t
from trew_b200 import synth
lib = t.load(sys.argv[1])
for mn, mx in [(5, 32), (3, 64)]:
    reads = synth.adversarial_short(7 + mx, 500, max_unit=mx, lengths=[150, 161, 4 * mx - 1, 60])
    reads += [b"", b"A", b"N" * 160, b"TTAGGG" * 26 + b"TTAG"]
    t.compare(lib, 0, reads, None, mn, mx, min_units=1)
    r1, r2 = synth.adversarial_pairs(9 + mx, 400, read_len=160, max_unit=mx, truncate_mate2=0.2)
    t.compare(lib, 1, r1, r2, mn, mx, min_units=0)
t.compare(lib, 2, synth.adversarial_long(11, 60, min_len=140, max_len=4000), None, 5, 32, 150, min_units=1)
print("sanitizer run clean")
