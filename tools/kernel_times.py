#!/usr/bin/env python3
"""Per-kernel device times of the scan pipeline under torch.profiler (CUDA activities): one device-resident batch of the
bench shape (tools/profile_scan.py's defaults, 25 M reads), scanned a few times after a warm-up.

    python tools/kernel_times.py [reads] [scans] [min_mer] [max_mer] [mode 0 short / 1 pair] [read_len]

Prints one line per kernel: launches, total and per-scan milliseconds, sorted by total time.  TREW_B200_LIB selects the
library, so two builds can be compared by running the script once per library.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from trew_b200 import api  # noqa: E402

reads = int(sys.argv[1]) if len(sys.argv) > 1 else 25_000_000
scans = int(sys.argv[2]) if len(sys.argv) > 2 else 5
mn = int(sys.argv[3]) if len(sys.argv) > 3 else 5
mx = int(sys.argv[4]) if len(sys.argv) > 4 else 32
mode = int(sys.argv[5]) if len(sys.argv) > 5 else api.MODE_SHORT
read_len = int(sys.argv[6]) if len(sys.argv) > 6 else 150

torch.cuda.init()
with api.DeviceContext(mode, mn, mx) as ctx:
    h = ctx.synth_resident(1, reads, read_len, tel_ppm=10000, half_ppm=2000, n_ppm=1000, sub_ppm=10000)
    for _ in range(2):          # warm-up: first launches load the kernels
        ctx.scan_resident(h)
    ctx.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(scans):
            ctx.scan_resident(h)
        ctx.sync()
    ctx.free_resident(h)

rows = {}
for ev in prof.events():
    if ev.device_type != torch.autograd.DeviceType.CUDA:
        continue
    n, t = rows.get(ev.name, (0, 0.0))
    rows[ev.name] = (n + 1, t + ev.time_range.elapsed_us() / 1000.0)
print("lib %s  reads %d  scans %d  min_mer %d  max_mer %d  mode %d  len %d" %
      (os.path.basename(os.path.dirname(api.LIB_PATH)) + "/" + os.path.basename(api.LIB_PATH), reads, scans, mn, mx, mode, read_len))
print("%8s %10s %10s  %s" % ("launches", "total_ms", "ms/scan", "kernel"))
for name, (n, t) in sorted(rows.items(), key=lambda kv: -kv[1][1]):
    print("%8d %10.3f %10.3f  %s" % (n, t, t / scans, name[:140]))
