"""Reads whose windows run from 161 up to the 1023-base limit.  TEST INFRASTRUCTURE ONLY (seeded, deterministic).

Above 160 bases only the warp-per-survivor exact kernel decides a unit (trew_exact_kernel in scan_kernels.cu): paired
reads longer than 160 bases, short reads of 161..1000 bases and every long-read slice longer than 160 bases.  Its window
is 32 lanes x 32 bits, at most 1023 bases.  This corpus puts reads on the lengths where that code changes behaviour --
the thread/warp split, the whole-read probe, the filter variants (probe_filter<5>, <8>, pass-through), the screen's
first levels, the 1023-base window -- for short, paired and long configurations, and adds constructed windows, each
certified with the oracle's per-period statistics:

  limit_10bit    a 3-base repeat over a whole 1023-base window at MIN_MER 3: T = M = 1021 at k = 3, two short of the
                 10-bit fields of bound_k and of eval_k's packed result (and a 5-base repeat at MIN_MER 5)
  many_classes   a window of 1023 bases whose target period has >= 300 rotation classes (eval_k's hash holds hundreds
                 of runs, the warp emits hundreds of distinct keys)
  few_windows    N's spaced so that a period of a 1023-base window keeps <= 32 valid windows spread over many lanes
                 (comp_bound's case)
  few_runs       clean repeats of >= 511 bases whose target period has <= 12 match-bit runs (eval_k's serial path)
  margin_edge    edges.margin_pair windows of 256..1023 bases: margin 0 and its -1 twin against LOW

Every unit carries `regimes`: the constructed regime, if any, and the branches its geometry reaches (branch_tags).
"""
from __future__ import annotations

import random
from typing import Dict, List, Sequence, Tuple

import numpy as np

from oracle import edges
from oracle.oracle import Oracle
from trew_b200 import synth

MAX_WINDOW = 1023        # 32 lanes x 32 bits (scan_kernels.cuh kMaxWindow)
THREAD_MAX_READ = 160    # exact_thread.cuh kMaxRead: longer units go to the warp kernel
SERIAL_MAX_RUNS = 12     # scan_kernels.cu kSerialMaxRuns

SLICES = (64, 128, 159, 160, 161, 255, 256, 300, 511, 512)

# name -> (mode, MIN_MER, MAX_MER, LOW, HIGH, SLICE); mode 0 short, 1 paired, 2 long
CONFIGS: Dict[str, Tuple[int, int, int, float, float, int]] = {
    "short_5_32": (0, 5, 32, 0.5, 0.8, 150),
    "short_3_64": (0, 3, 64, 0.5, 0.8, 150),
    "short_12_40": (0, 12, 40, 0.5, 0.8, 150),
    "short_035_06": (0, 5, 32, 0.35, 0.6, 150),
    "pair_5_32": (1, 5, 32, 0.5, 0.8, 150),
    "pair_3_64": (1, 3, 64, 0.5, 0.8, 150),
    "pair_12_40": (1, 12, 40, 0.5, 0.8, 150),
}
for _sl in SLICES:
    CONFIGS["long_5_32_s%d" % _sl] = (2, 5, 32, 0.5, 0.8, _sl)
for _sl in SLICES:
    if _sl >= 128:
        CONFIGS["long_3_64_s%d" % _sl] = (2, 3, 64, 0.5, 0.8, _sl)

REGIMES = ("limit_10bit", "many_classes", "few_windows", "few_runs", "margin_edge")

PAIR_EQUAL = (161, 200, 250, 251, 300, 301, 511, 512, 513, 1022, 1023)
# min(n1, n2) on each side of 4 * MAX_MER at 3 64 (256); a 1023-base mate whose partner is short is scanned whole
PAIR_UNEQUAL = ((160, 161), (150, 300), (1023, 40), (1023, 255), (1023, 256))
PAIR_TRUNCATED = (300, 1023)   # mate 2 cut to a third .. all of the mate length


def lengths(name: str) -> List:
    """the length keys of a configuration: read lengths (short, long), (n1, n2) or ("trunc", n) (paired)"""
    mode, mn, mx, _, _, sl = CONFIGS[name]
    if mode == 0:
        return sorted({159, 160, 161, 4 * mx - 1, 4 * mx, 190, 191, 318, 319, 320, 510, 511, 512, 513, 700, 999, 1000})
    if mode == 1:
        return [(n, n) for n in PAIR_EQUAL] + list(PAIR_UNEQUAL) + [("trunc", n) for n in PAIR_TRUNCATED]
    out = [sl - 1, sl, 2 * sl - 1, 2 * sl, 3 * sl - 1, "4-20kb"]
    if sl == 2 * mx:
        out.append("50-200kb")   # hundreds to thousands of slices: the walks and their per-warp scratch
    return out


class Unit:
    __slots__ = ("mates", "length", "regimes")

    def __init__(self, mates, length, regimes):
        self.mates, self.length, self.regimes = list(mates), length, set(regimes)


def branch_tags(cfg, mates: Sequence[bytes]) -> List[str]:
    """the branches a unit's geometry reaches: exact kernel, probe windows and the filter variant each one needs"""
    mode, mn, mx, _, _, sl = cfg
    n1, n2 = len(mates[0]), len(mates[-1])
    t = []
    if mode == 2:
        if n1 < sl:
            return ["slice_dropped"]
        t.append("single_slice" if n1 < 2 * sl else "multi_slice")
        if n1 // sl >= 300:
            t.append("hundreds_of_slices")
        if sl > edges.FAST_MAX_WL_LONG:
            t.append("screen_skipped")
    else:
        t.append("thread" if max(n1, n2) <= THREAD_MAX_READ else "warp")
        if mode == 1 and n1 != n2:
            t.append("unequal_mates")
    for mate, st, wl, k0, k1 in edges.unit_probes(mode, mn, mx, sl, n1, n2):
        if mode != 2 and st == 0 and wl == len(mates[mate]):
            t.append("whole_read_probe")
        if wl + 1 <= 96:
            t.append("probe_filter3")
        elif wl + 1 <= 160:
            t.append("probe_filter5")
        elif wl + 1 <= 256:
            t.append("probe_filter8")
        else:
            t.append("pass_through")
        if wl >= 512:
            t.append("window_512_plus")
        if wl == MAX_WINDOW:
            t.append("window_1023")
        if mode == 2 and wl > THREAD_MAX_READ:
            t.append("slice_over_160")
    return sorted(set(t))


def match_runs(seq: bytes, st: int, nd: int, k: int) -> int:
    """eval_k's run count of period k over seq[st..nd]: maximal runs of valid k-windows i, i+1, ... with base i == base i+k"""
    w = np.frombuffer(seq[st:nd + 1].upper(), dtype=np.uint8)
    nwin = len(w) - k + 1
    if nwin <= 0:
        return 0
    bad = np.concatenate([[0], np.cumsum(~np.isin(w, np.frombuffer(b"ACGT", np.uint8)))])
    i = np.arange(nwin)
    valid = (bad[i + k] - bad[i]) == 0
    link = np.zeros(nwin, dtype=bool)
    link[:-1] = valid[:-1] & valid[1:] & (w[:nwin - 1] == w[k:k + nwin - 1])
    starts = valid & ~np.concatenate([[False], link[:-1]])
    return int(starts.sum())


# ---------------------------------------------------------------- reads at the table's lengths

def _seed(rng: random.Random) -> int:
    return rng.randrange(1 << 30)


def length_units(rng: random.Random, name: str, per: int) -> List[Unit]:
    cfg = CONFIGS[name]
    mode, mn, mx, _, _, sl = cfg
    units: List[Unit] = []
    for key in lengths(name):
        if mode == 0:
            reads = synth.adversarial_short(_seed(rng), per, max_unit=mx, lengths=[key])
            units += [Unit([r], key, branch_tags(cfg, [r])) for r in reads]
        elif mode == 1:
            if key[0] == "trunc":
                r1, r2 = synth.adversarial_pairs(_seed(rng), per, read_len=key[1], max_unit=mx, truncate_mate2=1.0)
            else:
                n1, n2 = key
                r1, r2 = synth.adversarial_pairs(_seed(rng), per, read_len=max(n1, n2), max_unit=mx)
                r1, r2 = [r[:n1] for r in r1], [r[:n2] for r in r2]
            units += [Unit([a, b], key, ["truncated_mate"] * (key[0] == "trunc") + branch_tags(cfg, [a, b])) for a, b in zip(r1, r2)]
        else:
            if key == "4-20kb":
                reads = synth.adversarial_long(_seed(rng), max(2, per // 2), min_len=4000, max_len=20000, max_unit=mx)
            elif key == "50-200kb":
                reads = synth.adversarial_long(_seed(rng), 2, min_len=50000, max_len=200000, max_unit=mx)
            else:
                reads = synth.adversarial_long(_seed(rng), per, min_len=key, max_len=key, max_unit=mx)
            units += [Unit([r], key, branch_tags(cfg, [r])) for r in reads]
    return units


# ---------------------------------------------------------------- constructed regimes

def _rand(rng: random.Random, n: int) -> bytes:
    return bytes(rng.choice(b"ACGT") for _ in range(n))


def _unit(rng: random.Random, p: int) -> bytes:
    """a primitive unit of p bases (no shorter period), so that a repeat of it has its first period at p"""
    while True:
        u = _rand(rng, p)
        if all(u != (u[:d] * (p // d)) for d in range(1, p) if p % d == 0):
            return u


def _as_unit(cfg, window: bytes, rng: random.Random) -> Tuple[List[bytes], Tuple[int, int]]:
    """a unit of this configuration whose first probe is `window` whole; (mates, (st, nd) of the window in mate 1).  Long
    mode: a single-slice read.  Paired mode: the partner is shorter than 4 * MIN_MER, so mate 1 is scanned whole, with k
    from MIN_MER up."""
    mode, mn, mx, _, _, sl = cfg
    mates = [window, _rand(rng, 2 * mn + rng.randint(0, 1))] if mode == 1 else [window]
    return mates, (0, len(window) - 1)


def _probe_k(cfg, mates) -> Tuple[int, int]:
    mode, mn, mx, _, _, sl = cfg
    p = edges.unit_probes(mode, mn, mx, sl, len(mates[0]), len(mates[-1]))
    return p[0][3], p[0][4]


def limit_units(o: Oracle, rng: random.Random, cfg) -> List[Unit]:
    """a repeat of a primitive unit of MIN_MER bases over a whole 1023-base window: T = M = 1023 - MIN_MER + 1.  The units
    cover the four hi/lo parity signatures, so the 10-bit fields of bound_k's buckets all reach T."""
    mode, mn, mx, _, _, sl = cfg
    units, seen = [], set()
    tries = 0
    while len(seen) < 4 and tries < 400:
        tries += 1
        u = _unit(rng, mn)
        sig = (sum(b in b"AC" for b in u) & 1, sum(b in b"AG" for b in u) & 1)   # hi = A|C, lo = A|G (T 0, G 1, C 2, A 3)
        if sig in seen:
            continue
        w = (u * (MAX_WINDOW // mn + 1))[:MAX_WINDOW]
        mates, (st, nd) = _as_unit(cfg, w, rng)
        k0, k1 = _probe_k(cfg, mates)
        T, M, _, _ = o.period_stats(w, st, nd, mn)
        if k0 != mn or (T, M) != (MAX_WINDOW - mn + 1, MAX_WINDOW - mn + 1):
            continue
        seen.add(sig)
        units.append(Unit(mates, MAX_WINDOW, ["limit_10bit"] + branch_tags(cfg, mates)))
    return units


def many_class_units(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """a period-MAX_MER unit over ~530 bases, then random bases, in a 1023-base window: accepted at k = MAX_MER with
    hundreds of rotation classes"""
    mode, mn, mx, _, _, sl = cfg
    units, tries = [], 0
    while len(units) < count and tries < 40 * count:
        tries += 1
        p = rng.choice([mx, mx - 1, mx - 2]) if mx <= 32 else rng.choice([32, 40, 48])
        rep = rng.randint(515, 560)
        w = (_unit(rng, p) * (rep // p + 1))[:rep] + _rand(rng, MAX_WINDOW - rep)
        mates, (st, nd) = _as_unit(cfg, w, rng)
        k0, k1 = _probe_k(cfg, mates)
        th, tl = o.k_mer_check(w, st, nd, k0, k1)[:2]
        k = tl or th
        if not k:
            continue
        T, M, _, ncls = o.period_stats(w, st, nd, k)
        if ncls >= 300 and match_runs(w, st, nd, k) > SERIAL_MAX_RUNS:
            units.append(Unit(mates, MAX_WINDOW, ["many_classes"] + branch_tags(cfg, mates)))
    return units


def few_window_units(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """a repeat of period p with an N every g bases (g = p + 1 or p + 2): period p keeps one or two valid windows per
    gap, <= 32 in all, spread over the lanes of a 1023-base window"""
    mode, mn, mx, _, _, sl = cfg
    units, tries = [], 0
    while len(units) < count and tries < 40 * count:
        tries += 1
        p = rng.randint(max(mn, mx - 8), mx)
        g = p + rng.choice([1, 2])
        w = bytearray((_unit(rng, p) * (MAX_WINDOW // p + 1))[:MAX_WINDOW])
        for q in range(rng.randrange(g), MAX_WINDOW, g):
            w[q] = ord("N")
        w = bytes(w)
        mates, (st, nd) = _as_unit(cfg, w, rng)
        k0, k1 = _probe_k(cfg, mates)
        few = [k for k in range(k0, k1 + 1) if 0 < o.period_stats(w, st, nd, k)[0] <= 32]
        if p not in few:
            continue
        starts = [i for i in range(MAX_WINDOW - p + 1) if b"N" not in w[i:i + p]]
        if len({i // 32 for i in starts}) >= 12:
            units.append(Unit(mates, MAX_WINDOW, ["few_windows"] + branch_tags(cfg, mates)))
    return units


def few_run_units(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """clean repeats (a few substitutions at most) over a window of >= 511 bases whose target period has <= 12 runs"""
    mode, mn, mx, _, _, sl = cfg
    units, tries = [], 0
    while len(units) < count and tries < 40 * count:
        tries += 1
        p = rng.randint(mn, mx)
        if mode == 0:
            n = rng.choice([1000, 999])        # halves of 500, the whole read a target window
        elif mode == 1:
            n = rng.choice([1022, 1023])       # segments of 511 and 512
        else:
            n = rng.randint(max(sl, 511), 2 * sl - 1)
        r = bytearray((_unit(rng, p) * (n // p + 1))[:n])
        for _ in range(rng.randint(0, 3)):
            r[rng.randrange(n)] = rng.choice(b"ACGT")
        r = bytes(r)
        mates = [r, bytes(synth.revcomp(r))] if mode == 1 else [r]
        probes = edges.unit_probes(mode, mn, mx, sl, len(mates[0]), len(mates[-1]))
        _, st, wl, k0, k1 = probes[0]
        th, tl = o.k_mer_check(r, st, st + wl - 1, k0, k1)[:2]
        if tl and wl >= 500 and match_runs(r, st, st + wl - 1, tl) <= SERIAL_MAX_RUNS:
            units.append(Unit(mates, n, ["few_runs"] + branch_tags(cfg, mates)))
    return units


MARGIN_WINDOWS = {0: (256, 300, 500), 1: (256, 300, 500, 511), 2: (600, 800, 1023)}


def margin_units(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """edges.margin_pair at long window lengths: a window at margin 0 against LOW and its twin at -1"""
    mode, mn, mx, low, _, sl = cfg
    units = []
    for wl in MARGIN_WINDOWS[mode]:
        if mode == 2 and not sl <= wl < 2 * sl:
            continue
        got, tries = 0, 0
        while got < count and tries < 20 * count:
            tries += 1
            p = rng.choice([p for p in (6, 7, 13, 24, 31, 32, 40, 64, 3) if mn <= p <= mx])
            r = edges.margin_pair(o, rng, cfg, wl, p, rng.choice([0, 2]), low)
            if r is None or max(len(m) for m in r[0] + r[1]) > (1000 if mode == 0 else MAX_WINDOW if mode == 1 else 2 * sl - 1):
                continue
            got += 1
            for mates in r[:2]:
                units.append(Unit(mates, wl, ["margin_edge"] + branch_tags(cfg, mates)))
    return units


def corpus(name: str, seed: int = 1, per: int = 8) -> List[Unit]:
    """the long-window corpus of one configuration: `per` reads at each length of the table, then the constructed
    regimes that apply to it"""
    cfg = CONFIGS[name]
    mode, mn, mx, low, high, sl = cfg
    o = Oracle(mn, mx, low, high, slice_len=sl)
    rng = random.Random(seed * 1000003 + sum(map(ord, name)))
    units = length_units(rng, name, per)
    window_fits = mode != 2 or sl == 512   # a 1023-base window: a whole mate or a single slice at SLICE 512
    if window_fits and mn in (3, 5) and mode != 0:
        units += limit_units(o, rng, cfg)
    if window_fits and mode == 2:
        units += many_class_units(o, rng, cfg, 3)
        units += few_window_units(o, rng, cfg, 4)
    if name in ("short_5_32", "pair_5_32", "pair_3_64", "long_5_32_s512", "long_3_64_s512", "long_5_32_s300"):
        units += few_run_units(o, rng, cfg, 4)
    if name in ("short_5_32", "pair_5_32", "pair_3_64", "long_5_32_s512"):
        units += margin_units(o, rng, cfg, 2)
    return units


def regime_counts(units: Sequence[Unit]) -> Dict[str, int]:
    out: Dict[str, int] = {}
    for u in units:
        for r in u.regimes:
            out[r] = out.get(r, 0) + 1
    return dict(sorted(out.items()))


def scan_args(name: str, units: Sequence[Unit]):
    """(mode, reads1, reads2) for Oracle.scan / DeviceContext.submit_reads"""
    mode = CONFIGS[name][0]
    r1 = [u.mates[0] for u in units]
    r2 = [u.mates[1] for u in units] if mode == 1 else None
    return mode, r1, r2
