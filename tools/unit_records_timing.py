#!/usr/bin/env python3
"""What per-unit hit records cost on the bench shapes: device-resident synthetic batches (trew_synth_resident_ex, the
BASELINE.json shapes), scanned by one context without records and one with them, alternated.

    python tools/unit_records_timing.py [reps] [scans]

Per shape: scan Gbases/s of both contexts (CUDA events around `scans` scans of one batch, after a reset), records per unit
and their bytes, the time of the records call (device sort + sum + copy to the host, wall clock) and a check that the
records summed over units give the tables of finish().  Prints the card's name and power limit first."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from trew_b200 import api  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
scans = int(sys.argv[2]) if len(sys.argv) > 2 else 3
SYNTH = dict(tel_ppm=10000, half_ppm=2000, n_ppm=1000, sub_ppm=10000)
# name, mode, min_mer, max_mer, flavor, reads per batch, read length (BASELINE.json configs[1..3])
SHAPES = [("short_150", api.MODE_SHORT, 5, 32, 0, 25_000_000, 150), ("paired_2x150", api.MODE_PAIR, 5, 32, 1, 25_000_000, 150),
          ("long_15kb", api.MODE_LONG, 5, 32, 2, 200_000, 15000)]
CAP = 1 << 28


def keyed_sums(v):
    meta = v["table"].astype(np.uint64) << np.uint64(8) | v["k"].astype(np.uint64)
    order = np.lexsort((v["seq_lo"], v["seq_hi"], meta))
    m, h, lo, c = meta[order], v["seq_hi"][order], v["seq_lo"][order], v["count"][order].astype(np.uint64)
    head = np.ones(len(m), dtype=bool)
    head[1:] = (m[1:] != m[:-1]) | (h[1:] != h[:-1]) | (lo[1:] != lo[:-1])
    idx = np.flatnonzero(head)
    return m[idx], h[idx], lo[idx], np.add.reduceat(c, idx) if len(c) else c


def timed_scans(ctx, h):
    ctx.reset()
    ctx.timer_start()
    for _ in range(scans):
        ctx.scan_resident(h)
    return ctx.timer_stop()


q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print("gpu:", q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown")
print("%-13s %9s %9s %8s %11s %11s %10s %9s  %s" % ("shape", "off_Gb/s", "on_Gb/s", "on/off", "recs/unit", "rec_MB", "finish_ms", "units", "identity"))
for name, mode, mn, mx, flavor, n_reads, rl in SHAPES:
    off = api.DeviceContext(mode, mn, mx)
    on = api.DeviceContext(mode, mn, mx)
    on.enable_unit_records(CAP)
    h_off = off.synth_resident(1, n_reads, rl, flavor=flavor, **SYNTH)
    h_on = on.synth_resident(1, n_reads, rl, flavor=flavor, **SYNTH)
    for c, h in ((off, h_off), (on, h_on)):   # warm-up
        timed_scans(c, h)
    t_off, t_on = [], []
    for _ in range(reps):
        t_off.append(timed_scans(off, h_off))
        t_on.append(timed_scans(on, h_on))
    bases = float(n_reads) * rl * scans
    t0 = time.perf_counter()
    recs = on.unit_records()
    fin_ms = (time.perf_counter() - t0) * 1e3
    tables = on.finish_view().copy()
    plain = off.finish_view().copy()
    a, b = keyed_sums(recs), keyed_sums(tables)
    ok = all(np.array_equal(x, y) for x, y in zip(a, b)) and np.array_equal(tables, plain)
    units = (n_reads // 2 if mode == api.MODE_PAIR else n_reads) * scans
    print("%-13s %9.1f %9.1f %8.3f %11.4f %11.1f %10.1f %9d  %s" % (
        name, bases / (np.median(t_off) * 1e6), bases / (np.median(t_on) * 1e6), np.median(t_off) / np.median(t_on), len(recs) / units,
        len(recs) * 32 / 1e6, fin_ms, units, "records sum to the tables, tables equal with records off" if ok else "MISMATCH"))
    print("   scan ms off %s  on %s" % (" ".join("%.2f" % t for t in t_off), " ".join("%.2f" % t for t in t_on)))
    for c, h in ((off, h_off), (on, h_on)):
        c.free_resident(h)
        c.close()
