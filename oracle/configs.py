"""A seeded grid of scan configurations, with a corpus per configuration.  TEST INFRASTRUCTURE ONLY (deterministic).

The command line takes any 3 <= MIN_MER <= MAX_MER <= 64, 0 < LOW <= HIGH <= 1 and, in long mode, any
2 * MAX_MER <= SLICE_LENGTH <= 512.  The device code changes path at points between the configurations the other corpora
use: k = 16 / 17 (canon64's 32-bit loop), 31 / 32 / 33 (64- vs 128-bit units, fast_span<0> / <1>), MAX_MER 37 / 38 and
40 / 41 (a 150-base read's whole-read probe, the 160-base thread limit), 63 / 64 (probe_is_fast, fast_span_long<2>,
HD_BLK64), the MIN_MER guards of unit_probes, the decide kernel's variant at SLICE 47 / 48, 79 / 80, 128 / 129, 159 / 160,
and the baselines' threshold tables.  CONFIGS names the boundary points first, then a seeded set of random points.

Every unit is derived from its configuration and carries `regimes`: the constructed regime it was built for, and the
branches its geometry reaches (long_windows.branch_tags).  Constructed units are certified with the oracle's per-period
statistics and dropped when the certificate disagrees:

  len_<key>      reads of the lengths where the routing changes: 2 MIN - 1, 2 MIN, 4 MIN - 1, 4 MIN, 4 MAX - 1, 4 MAX,
                 150, 160, 161 (short); pairs whose shorter mate sits on each side of 4 MAX; long reads of SL - 1 .. 3 SL - 1
                 bases and a few kb (tens of kb at small SLICE)
  period         a repeat whose accepted period is exactly a boundary period (MIN, MAX, 16, 17, 32, 33, 63, 64)
  whole64        MAX_MER 64: a read of 128..159 bases whose only accepted period is 64, in the whole-read probe
  divisor        a repeat of period p whose multiples (16 -> 32 -> 64, 21 -> 42 -> 63, 32 -> 64) would each pass but are
                 blocked by the accepted p
  margin_low / margin_high
                 edges.margin_pair windows at margin 0 and -1 against LOW / HIGH (regimes margin_*_0 and margin_*_-1)
  n_per_half     one N in each half (each probe window) of a read
  few_windows    N's spaced so that a period keeps at most 32 valid windows
  dense          at LOW <= 0.2: uniform random reads, most of which emit dozens of keys of count 1
"""
from __future__ import annotations

import random
from typing import Dict, List, Sequence, Tuple

from oracle import edges
from oracle import long_windows as lw
from oracle.oracle import Oracle
from trew_b200 import synth

Config = Tuple[int, int, int, float, float, int]   # (mode, MIN_MER, MAX_MER, LOW, HIGH, SLICE); mode 0 short, 1 paired, 2 long

MAX_SHORT, MAX_PAIR = 1000, 1023     # the longest read (mate) submit_chunk accepts
BOUNDARY_MAX = (3, 16, 17, 31, 32, 33, 37, 38, 40, 41, 63, 64)
BOUNDARY_PERIODS = (16, 17, 32, 33, 63, 64)
DIVISOR_CHAINS = ((16, 32, 64), (21, 42, 63), (32, 64))
BASELINES = ((0.05, 0.1), (0.1, 0.2), (0.15, 0.8), (0.2, 1.0), (0.5, 1.0), (0.7, 0.7), (1.0, 1.0), (1 / 3, 2 / 3))
NEXT_ABOVE = (0.5000000000000001, 0.30000000000000004)   # math.nextafter(0.5, 1), math.nextafter(0.3, 1)
DENSE_LOW = 0.2
MARGIN_LEAST = 0.3


def _mid_min(mx: int) -> int:
    """a MIN_MER below MAX_MER whose 2 * MIN / 4 * MIN fall on common read lengths (76, 80, 152, 160), or 10 (20 / 40)"""
    for m in (40, 38, 19):
        if m < mx:
            return m
    return 10 if 10 < mx else mx


def _grid() -> Dict[str, Config]:
    c: Dict[str, Config] = {}
    for mx in BOUNDARY_MAX:
        for mn in sorted({3, mx, _mid_min(mx)}):
            c["short_%d_%d" % (mn, mx)] = (0, mn, mx, 0.5, 0.8, 150)
    for mn, mx in ((3, 16), (3, 17), (16, 17), (3, 33), (31, 32), (19, 37), (38, 38), (3, 41), (40, 41), (3, 63), (64, 64)):
        c["pair_%d_%d" % (mn, mx)] = (1, mn, mx, 0.5, 0.8, 150)
    for mn, mx in ((3, 16), (17, 17), (3, 33), (32, 32), (3, 64), (63, 64)):
        c["long_%d_%d" % (mn, mx)] = (2, mn, mx, 0.5, 0.8, 150)
    for low, high in BASELINES + tuple((b, b) for b in NEXT_ABOVE):
        tag = "%.17g_%.17g" % (low, high)
        c["short_5_32_" + tag] = (0, 5, 32, low, high, 150)
        c["pair_5_32_" + tag] = (1, 5, 32, low, high, 150)
    for low, high in ((0.05, 0.1), (0.1, 0.2), (1.0, 1.0), (1 / 3, 2 / 3), (NEXT_ABOVE[1], NEXT_ABOVE[1])):
        tag = "%.17g_%.17g" % (low, high)
        c["short_3_64_" + tag] = (0, 3, 64, low, high, 150)
        c["pair_3_64_" + tag] = (1, 3, 64, low, high, 150)
        c["long_5_32_" + tag] = (2, 5, 32, low, high, 150)
    c["long_3_3_s6"] = (2, 3, 3, 0.5, 0.8, 6)
    for mx in (5, 20, 32, 64):
        c["long_3_%d_s%d" % (mx, 2 * mx)] = (2, 3, mx, 0.5, 0.8, 2 * mx)
    for sl in (47, 48):   # SLICE >= 2 MAX_MER: at 5 32 these are refused
        c["long_5_23_s%d" % sl] = (2, 5, 23, 0.5, 0.8, sl)
    for sl in (79, 80, 128, 129, 159, 160):
        c["long_5_32_s%d" % sl] = (2, 5, 32, 0.5, 0.8, sl)
    c["long_3_64_s512"] = (2, 3, 64, 0.5, 0.8, 512)
    c["long_5_32_s64_0.1_0.2"] = (2, 5, 32, 0.1, 0.2, 64)
    rng = random.Random(20261022)
    for i in range(20):
        mode = i % 3
        mn, mx = sorted((rng.randint(3, 64), rng.randint(3, 64)))
        low, high = sorted((1.0 - rng.random(), 1.0 - rng.random()))   # (0, 1]
        sl = rng.randint(2 * mx, 512) if mode == 2 else 150
        c["random_%02d" % i] = (mode, mn, mx, low, high, sl)
    return c


CONFIGS: Dict[str, Config] = _grid()


class Unit:
    __slots__ = ("mates", "regimes")

    def __init__(self, mates, regimes):
        self.mates, self.regimes = list(mates), set(regimes)


def oracle_for(cfg: Config) -> Oracle:
    mode, mn, mx, low, high, sl = cfg
    return Oracle(mn, mx, low, high, slice_len=sl)


def _rand(rng: random.Random, n: int) -> bytes:
    return bytes(rng.choice(b"ACGT") for _ in range(n))


def _fits(cfg: Config, mates: Sequence[bytes]) -> bool:
    mode = cfg[0]
    if mode == 0:
        return 1 <= len(mates[0]) <= MAX_SHORT
    if mode == 1:
        return all(1 <= len(m) <= MAX_PAIR for m in mates)
    return len(mates[0]) >= 1


def _unit(cfg: Config, mates: Sequence[bytes], regimes: Sequence[str]) -> Unit:
    return Unit(mates, list(regimes) + lw.branch_tags(cfg, mates))


def _mates(cfg: Config, rng: random.Random, r: bytes) -> List[bytes]:
    """r as a unit: a read, or mate 1 of a pair whose mate 2 is r's reverse complement (both mates probed alike)"""
    return [r, synth.revcomp(r)] if cfg[0] == 1 else [r]


# ---------------------------------------------------------------- read lengths

def lengths(cfg: Config) -> List:
    """the length keys of a configuration: n (short, long), (n1, n2) (paired), or "kb" (long)"""
    mode, mn, mx, _, _, sl = cfg
    if mode == 0:
        return sorted({n for n in (2 * mn - 1, 2 * mn, 4 * mn - 1, 4 * mn, 4 * mx - 1, 4 * mx, 150, 160, 161) if 1 <= n <= MAX_SHORT})
    if mode == 1:
        out = {(150, 150), (150, 140), (160, 161), (2 * mn, 2 * mn + 3), (2 * mn - 1, 150)}
        for n in (4 * mx - 1, 4 * mx):                           # min(n1, n2) on each side of 4 MAX, either mate shorter
            out |= {(n, n), (n, n + 7), (n + 7, n)}
        return sorted(p for p in out if 1 <= min(p) and max(p) <= MAX_PAIR)
    return [sl - 1, sl, 2 * sl - 1, 2 * sl, 3 * sl - 1, "kb"]


def length_units(rng: random.Random, cfg: Config, per: int) -> List[Unit]:
    mode, mn, mx, _, _, sl = cfg
    units: List[Unit] = []
    seed = lambda: rng.randrange(1 << 30)
    for key in lengths(cfg):
        tag = "len_%s" % (key if not isinstance(key, tuple) else "%d_%d" % key)
        if mode == 0:
            reads = synth.adversarial_short(seed(), per, max_unit=mx, lengths=[key])
            units += [_unit(cfg, [r], [tag]) for r in reads]
        elif mode == 1:
            n1, n2 = key
            r1, r2 = synth.adversarial_pairs(seed(), per, read_len=max(n1, n2), max_unit=mx)
            units += [_unit(cfg, [a[:n1], b[:n2]], [tag]) for a, b in zip(r1, r2) if len(a) >= n1 and len(b) >= n2]
        elif key == "kb":
            lo, hi = (20000, 40000) if sl <= 16 else (3000, 8000)   # thousands of slices at small SLICE
            reads = synth.adversarial_long(seed(), max(2, per // 8), min_len=lo, max_len=hi, max_unit=mx)
            units += [_unit(cfg, [r], [tag]) for r in reads]
        else:
            reads = synth.adversarial_long(seed(), per // 2, min_len=key, max_len=key, max_unit=mx)
            units += [_unit(cfg, [r], [tag]) for r in reads]
    return units


# ---------------------------------------------------------------- repeats at a boundary period

def primitive(rng: random.Random, p: int) -> bytes:
    return lw._unit(rng, p)


def accepted(o: Oracle, seq: bytes, probe) -> Tuple[int, int]:
    """(th, tl) of k_mer_check over one probe window"""
    _, st, wl, k0, k1 = probe
    return o.k_mer_check(seq, st, st + wl - 1, k0, k1)[:2]


def _probes(cfg: Config, mates: Sequence[bytes]):
    mode, mn, mx, _, _, sl = cfg
    return edges.unit_probes(mode, mn, mx, sl, len(mates[0]), len(mates[-1]))


def period_lengths(cfg: Config, p: int) -> List[int]:
    """read lengths at which period p is in the k range of a probe"""
    mode, mn, mx, _, _, sl = cfg
    if mode == 2:
        return [sl + (sl - 1) // 3, 2 * sl - 1]
    out = [n for n in (4 * p, 4 * p + 3, 2 * p + 1, 3 * p, 150, 4 * mx - 1) if n >= 2 * mn]
    cap = MAX_SHORT if mode == 0 else MAX_PAIR
    return sorted({n for n in out if n <= cap})


def period_units(o: Oracle, rng: random.Random, cfg: Config) -> List[Unit]:
    """a repeat of a primitive unit of p bases, for each boundary period p in [MIN, MAX]: accepted at exactly p (tl or th)
    in a probe whose k range holds p"""
    mode, mn, mx, _, _, sl = cfg
    units: List[Unit] = []
    for p in sorted({mn, mx} | {q for q in BOUNDARY_PERIODS if mn <= q <= mx}):
        for n in period_lengths(cfg, p):
            for variant in range(2):
                r = (primitive(rng, p) * (n // p + 2))[:n]
                if variant:   # one substitution away from perfect
                    b = bytearray(r)
                    b[rng.randrange(n)] = rng.choice(b"ACGT")
                    r = bytes(b)
                mates = _mates(cfg, rng, r)
                if not _fits(cfg, mates):
                    continue
                if period_certified(o, cfg, mates, p):
                    units.append(_unit(cfg, mates, ["period", "period_%d" % p]))
    return units


def period_certified(o: Oracle, cfg: Config, mates, p: int) -> bool:
    return any(pr[3] <= p <= pr[4] and p in accepted(o, mates[pr[0]], pr) for pr in _probes(cfg, mates))


def whole64_units(o: Oracle, rng: random.Random, cfg: Config, count: int) -> List[Unit]:
    """MAX_MER 64: a read of 128..159 bases whose only period at LOW, in its whole-read probe, is 64 (the screen's
    fast_span_long<2>, the one span k = 64 reaches)"""
    mode, mn, mx, low, _, sl = cfg
    units: List[Unit] = []
    if mode == 2 or mx != 64 or mn > 64:
        return units
    tries = 0
    while len(units) < count and tries < 20 * count:
        tries += 1
        n = rng.randint(128, 159)
        r = (primitive(rng, 64) * 3)[:n]
        mates = _mates(cfg, rng, r)
        if whole64_certified(o, cfg, mates):
            units.append(_unit(cfg, mates, ["whole64"]))
    return units


def whole64_certified(o: Oracle, cfg: Config, mates) -> bool:
    low = cfg[3]
    probes = _probes(cfg, mates)
    whole = [pr for pr in probes if pr[1] == 0 and pr[2] == len(mates[pr[0]])]
    if not whole or not 128 <= len(mates[0]) <= 159:
        return False
    _, st, wl, k0, k1 = whole[0]
    if k1 != 64 or accepted(o, mates[0], whole[0])[1] != 64:
        return False
    for pr in probes:
        for k in range(pr[3], pr[4] + 1):
            if k == 64 and pr in whole:
                continue
            T, M, _, _ = o.period_stats(mates[pr[0]], pr[1], pr[1] + pr[2] - 1, k)
            if T and M >= Oracle.need(T, low):
                return False
    return True


def divisor_units(o: Oracle, rng: random.Random, cfg: Config) -> List[Unit]:
    """a perfect repeat of period p (the first of a chain) over a probe whose k range holds p and at least one multiple"""
    mode, mn, mx, low, _, sl = cfg
    units: List[Unit] = []
    for chain in DIVISOR_CHAINS:
        p, top = chain[0], max([q for q in chain if q <= mx], default=0)
        if p < mn or top <= p:
            continue
        ns = [4 * top, 4 * top + 2, 2 * top + 2] if mode != 2 else [max(sl, 2 * top), 2 * sl - 1]
        for n in ns:
            r = (primitive(rng, p) * (n // p + 2))[:n]
            mates = _mates(cfg, rng, r)
            if _fits(cfg, mates) and divisor_certified(o, cfg, mates, chain):
                units.append(_unit(cfg, mates, ["divisor", "divisor_%d_%d" % (p, top)]))
    return units


def divisor_certified(o: Oracle, cfg: Config, mates, chain) -> bool:
    """p accepted; every multiple of the chain in the probe's k range passes LOW on its own (it is only blocked)"""
    low = cfg[3]
    for pr in _probes(cfg, mates):
        mult = [q for q in chain[1:] if pr[3] <= q <= pr[4]]
        if not mult or not pr[3] <= chain[0] <= pr[4]:
            continue
        if accepted(o, mates[pr[0]], pr)[1] != chain[0]:
            continue
        ok = True
        for q in mult:
            T, M, _, _ = o.period_stats(mates[pr[0]], pr[1], pr[1] + pr[2] - 1, q)
            ok = ok and T > 0 and M >= Oracle.need(T, low)
        if ok:
            return True
    return False


# ---------------------------------------------------------------- margins, N's, dense reads

def margin_units(o: Oracle, rng: random.Random, cfg: Config, count: int) -> List[Unit]:
    """edges.margin_pair against LOW and against HIGH: a read at margin 0 and its twin at -1"""
    mode, mn, mx, low, high, sl = cfg
    units: List[Unit] = []
    for name, B in (("low", low), ("high", high)):
        if name == "high" and high == low:
            continue
        got, tries = 0, 0
        while got < count and tries < 80 * count:
            tries += 1
            if mode == 2:
                wl = rng.randint(sl, 2 * sl - 1)
                p = rng.randint(mn, min(mx, wl // 2))
            else:
                wl = rng.randint(max(2 * mn, 10), max(2 * mn, min(159, MAX_SHORT // 2)))
                if rng.random() < 0.5:
                    wl = rng.randint(max(2 * mn, 10), max(2 * mn, 95))
                if wl // 2 < mn:
                    continue
                p = rng.randint(mn, min(mx, wl // 2))
            r = edges.margin_pair(o, rng, cfg, wl, p, rng.choice([0, 0, 1]), B)
            if r is None or not all(_fits(cfg, m) for m in r[:2]):
                continue
            got += 1
            for mates, m in ((r[0], 0), (r[1], -1)):
                units.append(_unit(cfg, mates, ["margin_%s" % name, "margin_%s_%d" % (name, m)]))
    return units


def n_units(o: Oracle, rng: random.Random, cfg: Config, count: int) -> List[Unit]:
    """one N in each probe window of a repeat read; and a repeat with an N every p + 1 or p + 2 bases, where period p
    keeps at most 32 valid windows"""
    mode, mn, mx, _, _, sl = cfg
    units: List[Unit] = []
    for i in range(count):
        if mode == 2:
            n = rng.choice([sl, 2 * sl - 1, 3 * sl - 1])
        else:
            n = rng.choice([n for n in (150, 4 * mx, 4 * mn) if n >= max(2 * mn, 4)])
        p = rng.randint(mn, max(mn, min(mx, n // 4)))
        mates = [bytearray(m) for m in _mates(cfg, rng, (primitive(rng, p) * (n // p + 2))[:n])]
        if i % 2 == 0:
            for m, st, wl, _, _ in _probes(cfg, mates):
                mates[m][st + rng.randrange(wl)] = ord("N")
            mates = [bytes(m) for m in mates]
            if _fits(cfg, mates) and n_certified(cfg, mates):
                units.append(_unit(cfg, mates, ["n_per_half"]))
        else:
            g = p + rng.choice([1, 2])
            for m in mates:
                for q in range(rng.randrange(g), n, g):
                    m[q] = ord("N")
            mates = [bytes(m) for m in mates]
            if _fits(cfg, mates) and few_certified(o, cfg, mates):
                units.append(_unit(cfg, mates, ["few_windows"]))
    return units


def n_certified(cfg: Config, mates) -> bool:
    pr = _probes(cfg, mates)
    return bool(pr) and all(b"N" in mates[m][st:st + wl] for m, st, wl, _, _ in pr)


def few_certified(o: Oracle, cfg: Config, mates) -> bool:
    for m, st, wl, k0, k1 in _probes(cfg, mates):
        for k in range(k0, k1 + 1):
            if 0 < o.period_stats(mates[m], st, st + wl - 1, k)[0] <= 32:
                return True
    return False


def dense_units(rng: random.Random, cfg: Config, count: int) -> List[Unit]:
    """uniform random reads (pairs) of 150 bases, or single-slice long reads"""
    mode, mn, mx, _, _, sl = cfg
    n = 2 * sl - 1 if mode == 2 else 150
    return [_unit(cfg, [_rand(rng, n)] + ([_rand(rng, n)] if mode == 1 else []), ["dense"]) for _ in range(count)]


# ---------------------------------------------------------------- the corpus

def corpus(name: str, seed: int = 1, per: int = 48) -> List[Unit]:
    """the corpus of one configuration: `per` reads at each length of the table, then the constructed regimes"""
    cfg = CONFIGS[name]
    mode, mn, mx, low, high, sl = cfg
    o = oracle_for(cfg)
    rng = random.Random(seed * 1000003 + sum(map(ord, name)))
    units = length_units(rng, cfg, per)
    units += period_units(o, rng, cfg)
    units += whole64_units(o, rng, cfg, 6)
    units += divisor_units(o, rng, cfg)
    units += margin_units(o, rng, cfg, 6)
    units += n_units(o, rng, cfg, 12)
    if low <= DENSE_LOW:
        units += dense_units(rng, cfg, 200)
    return units


def expected_regimes(name: str) -> Dict[str, int]:
    """regime -> the least number of units a configuration's corpus holds of it"""
    mode, mn, mx, low, high, sl = CONFIGS[name]
    out = {"n_per_half": 1, "few_windows": 1}
    for key in lengths(CONFIGS[name]):
        out["len_%s" % (key if not isinstance(key, tuple) else "%d_%d" % key)] = 1
    # below about 0.3 the random rest of a margin read (its other probes) clears the baseline itself
    if low >= MARGIN_LEAST:
        out["margin_low_0"] = out["margin_low_-1"] = 1
    if high != low and MARGIN_LEAST <= high < 1.0:
        out["margin_high_0"] = out["margin_high_-1"] = 1
    for p in {mn, mx} | {q for q in BOUNDARY_PERIODS if mn <= q <= mx}:
        out["period_%d" % p] = 1
    if mx == 64 and mode != 2 and low >= MARGIN_LEAST:
        out["whole64"] = 3
    for chain in DIVISOR_CHAINS:
        top = max([q for q in chain if q <= mx], default=0)
        if chain[0] >= mn and top > chain[0] and low >= MARGIN_LEAST:   # lower, a divisor of p is accepted and blocks p
            out["divisor_%d_%d" % (chain[0], top)] = 1
    if low <= DENSE_LOW:
        out["dense"] = 200
    return out


def certify(o: Oracle, cfg: Config, u: Unit) -> List[str]:
    """the regimes of u whose certificate does not hold (re-checked from scratch)"""
    bad = []
    mode, mn, mx, low, high, sl = cfg
    for r in u.regimes:
        if r.startswith("period_") and not period_certified(o, cfg, u.mates, int(r[7:])):
            bad.append(r)
        elif r == "whole64" and not whole64_certified(o, cfg, u.mates):
            bad.append(r)
        elif r.startswith("divisor_"):
            p, top = map(int, r.split("_")[1:])
            chain = next(c for c in DIVISOR_CHAINS if c[0] == p)
            if not divisor_certified(o, cfg, u.mates, chain):
                bad.append(r)
        elif r.startswith("margin_") and r.count("_") == 2:
            B = low if r.split("_")[1] == "low" else high
            if edges.unit_margin(o, cfg, u.mates, B) != int(r.split("_")[2]):
                bad.append(r)
        elif r == "n_per_half" and not n_certified(cfg, u.mates):
            bad.append(r)
        elif r == "few_windows" and not few_certified(o, cfg, u.mates):
            bad.append(r)
    return bad


def regime_counts(units: Sequence[Unit]) -> Dict[str, int]:
    return lw.regime_counts(units)


def scan_args(name: str, units: Sequence[Unit]):
    """(mode, reads1, reads2) for Oracle.scan / DeviceContext.submit_reads"""
    mode = CONFIGS[name][0]
    r1 = [u.mates[0] for u in units]
    r2 = [u.mates[1] for u in units] if mode == 1 else None
    return mode, r1, r2
