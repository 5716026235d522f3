"""Reads that sit exactly on an acceptance threshold.  TEST INFRASTRUCTURE ONLY (seeded, deterministic).

The scan filters (trew_b200/csrc/scan_kernels.cu: the screen kernel's first level, the decide kernel's levels) must never
turn away a probe window in which some period reaches LOW.  On random repeats almost every such window clears its
threshold by a wide margin, so a filter that is off by one at a comparison still passes them.  Here every read is built
so that, for a probe window as unit_probes defines the probes,

    margin = max over k in [k0, k1] of (M_k - need_LOW(T_k))

is exactly 0, and each has a twin at -1.  The construction is only a guess; every read is certified with the oracle's
per-period statistics (Oracle.period_stats) and dropped when the certificate disagrees.

Construction.  A probe window is periodic with a unit u of period p, except that one phase j of the unit takes up to four
different bases along the window: x in the first c unit copies, then y, z, w.  Every p-window holds exactly one phase-j
base, so the valid p-windows fall into at most four rotation classes (u with x, y, z or w at phase j), and the four
variants differ in the parities of their hi-bit and lo-bit counts: every level of the filters (parity, A-parity, counts
mod 4) puts each class into a bucket of its own, so at k = p each bucket count equals a class count.  The x-class count
is (j + 1) + (c - 1) * p, which is set to need_LOW(T).

Each read also carries `kills`: the comparisons of the filters that, made one tighter (`>=` -> `>`), would turn the whole
unit away.  They come from a plain restatement of the filter pipeline's bucket bounds (filter_bounds / unit_filter), so
a test can assert that the corpus holds reads on which such a mutation is visible.
"""
from __future__ import annotations

import math
import random
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from oracle.oracle import Oracle

CODES = {ord("T"): 0, ord("G"): 1, ord("C"): 2, ord("A"): 3}
LETTERS = b"TGCA"

# filter constants (scan_kernels.cu): the screen's fast first level covers windows of at most 95 bases (64 positions
# + E beyond), the long first level 96..159 bases (128 positions + E); the decide kernel asks its third level for periods
# with fewer than 48 valid windows and sends survivors with fewer than 36 to the warp kernel
FAST_MAX_WL, FAST_MAX_WL_LONG, MOD4_BELOW, THREAD_MIN_WINDOWS = 95, 159, 48, 36

# name -> (mode, MIN_MER, MAX_MER, LOW, HIGH, SLICE); mode 0 short, 1 paired, 2 long
CONFIGS: Dict[str, Tuple[int, int, int, float, float, int]] = {
    "short_5_32": (0, 5, 32, 0.5, 0.8, 150),
    "short_3_64": (0, 3, 64, 0.5, 0.8, 150),
    "short_12_40": (0, 12, 40, 0.5, 0.8, 150),
    "short_4_33": (0, 4, 33, 0.5, 0.8, 150),
    "short_035_06": (0, 5, 32, 0.35, 0.6, 150),
    "short_09_10": (0, 5, 32, 0.9, 1.0, 150),
    "short_05_05": (0, 5, 32, 0.5, 0.5, 150),
    "pair_5_32": (1, 5, 32, 0.5, 0.8, 150),
    "pair_3_64": (1, 3, 64, 0.5, 0.8, 150),
    "long_128": (2, 5, 32, 0.5, 0.8, 128),
    "long_150": (2, 5, 32, 0.5, 0.8, 150),
    # LOW = 0.55: (double)55 / 100 >= 0.55 although 0.55 * 100 rounds above 55 -- the case need_pre's slack is for
    "long_128_055": (2, 5, 32, 0.55, 0.8, 128),
}

MUTANTS = ("fast_entry", "decide_E", "decide_b1", "decide_U2", "mod4", "probe_filter_U2")


def encode(s: bytes) -> np.ndarray:
    return np.array([CODES.get(c & 0xDF, -1) for c in s], dtype=np.int8)


# ---------------------------------------------------------------- probes and margins

def unit_probes(mode: int, mn: int, mx: int, sl: int, n1: int, n2: int = 0) -> List[Tuple[int, int, int, int, int]]:
    """(mate, start, length, k0, k1) of the probe windows, as scan_kernels.cu:unit_probes forms them."""
    p = []
    if mode == 0:
        n = n1
        if n < 2 * mn:
            return p
        if n >= 4 * mn:
            kmax = min(n // 4, mx)
            p += [(0, 0, n // 2, mn, kmax), (0, n - (n + 1) // 2, (n + 1) // 2, mn, kmax)]
        if 4 * mx > n:
            p.append((0, 0, n, max(n // 4 + 1, mn), min(n // 2, mx)))
    elif mode == 1:
        n = min(n1, n2)
        if n < 2 * mn:
            return p
        if n >= 4 * mn:
            kmax = min(n // 4, mx)
            p += [(0, 0, n1 // 2, mn, kmax), (1, 0, n2 // 2, mn, kmax)]
        if 4 * mx > n:
            lo, hi = max(n // 4 + 1, mn), min(n // 2, mx)
            p += [(0, 0, n1, lo, hi), (1, 0, n2, lo, hi)]
    else:
        n = n1
        if n < sl:
            return p
        snum, bonus = n // sl, n % sl
        mid = (snum + 1) // 2
        l1 = sl + (bonus if mid == 1 else 0)
        p.append((0, 0, l1, mn, mx))
        if snum > 1:
            l2 = sl + (bonus if snum == mid else 0)
            p.append((0, n - l2, l2, mn, mx))
    return p


def probe_margin(o: Oracle, seq: bytes, st: int, wl: int, k0: int, k1: int, B: float) -> Optional[int]:
    """max over k of M_k - need_B(T_k); None when no period has a valid window"""
    best = None
    for k in range(k0, k1 + 1):
        T, M, _, _ = o.period_stats(seq, st, st + wl - 1, k)
        if T > 0:
            d = M - Oracle.need(T, B)
            best = d if best is None or d > best else best
    return best


def unit_margin(o: Oracle, cfg, mates: Sequence[bytes], B: Optional[float] = None) -> Optional[int]:
    mode, mn, mx, low, _, sl = cfg
    B = low if B is None else B
    best = None
    for mate, st, wl, k0, k1 in unit_probes(mode, mn, mx, sl, len(mates[0]), len(mates[-1])):
        d = probe_margin(o, mates[mate], st, wl, k0, k1, B)
        if d is not None and (best is None or d > best):
            best = d
    return best


# ---------------------------------------------------------------- the filters' bucket bounds, restated

def filter_bounds(codes: np.ndarray, st: int, wl: int, k: int):
    """(T, b64, E64, b128, E128, b1, b2, b3) of period k in window [st, st + wl): the largest parity bucket among the first
    64 / 128 window positions and the valid windows beyond them, and the largest bucket of the three levels over all
    valid windows (hi/lo parity; + A parity; hi/lo/A counts mod 4)."""
    w = codes[st:st + wl]
    nwin = wl - k + 1
    if nwin <= 0:
        return (0,) * 8
    z = np.zeros(1, np.int64)
    bad = np.concatenate([z, np.cumsum(w < 0)])
    wc = np.where(w < 0, 0, w).astype(np.int64)
    H = np.concatenate([z, np.cumsum(wc >> 1)])
    L = np.concatenate([z, np.cumsum(wc & 1)])
    A = np.concatenate([z, np.cumsum(wc == 3)])
    i = np.arange(nwin)
    ok = (bad[i + k] - bad[i]) == 0
    h, l, a = H[i + k] - H[i], L[i + k] - L[i], A[i + k] - A[i]
    s1 = (h & 1) | (l & 1) << 1
    s2 = s1 | (a & 1) << 2
    s3 = (h & 3) | (l & 3) << 2 | (a & 3) << 4

    def top(sig, sel, n):
        return int(np.bincount(sig[sel], minlength=n).max()) if sel.any() else 0
    T = int(ok.sum())
    f64, f128 = ok & (i < 64), ok & (i < 128)
    return (T, top(s1, f64, 4), T - int(f64.sum()), top(s1, f128, 4), T - int(f128.sum()), top(s1, ok, 4), top(s2, ok, 8),
            top(s3, ok, 64))


def probe_passes(cfg, codes: np.ndarray, probe, longest: int, mut: Optional[str] = None) -> Tuple[bool, int]:
    """(passes, t_hit): the screen kernel then the decide kernel on one probe, with the comparison `mut` made one tighter.
    t_hit = valid windows at the first period the decide kernel passes (1 << 20 when it is not the short decide)."""
    mode, _, _, low, _, sl = cfg
    _, st, wl, k0, k1 = probe
    if k1 < k0:
        return False, 1 << 20
    need = lambda T: Oracle.need(T, low)
    fb = {k: filter_bounds(codes, st, wl, k) for k in range(k0, k1 + 1)}
    clean = bool((codes[st:st + wl] >= 0).all())
    fast = wl <= FAST_MAX_WL and k1 <= 63 and k1 <= wl
    fast_long = wl <= FAST_MAX_WL_LONG and k1 <= 64 and k1 <= wl
    if not (mode == 2 and sl > FAST_MAX_WL_LONG) and clean:   # the screen kernel; a probe with an invalid base is deferred
        if fast:
            bump = 1 if mut == "fast_entry" else 0
            if not any(b[0] and b[1] + b[2] >= need(b[0]) + bump for b in fb.values()):
                return False, 1 << 20
        elif longest > FAST_MAX_WL and fast_long:
            if not any(b[0] and b[3] + b[4] >= need(b[0]) for b in fb.values()):
                return False, 1 << 20
    if fast:   # decide_short
        for k in range(k0, k1 + 1):
            T, b64, E64, _, _, b1, b2, b3 = fb[k]
            if T == 0:
                break
            n = need(T)
            if (b64 + E64 >= n + (mut == "decide_E") and b1 >= n + (mut == "decide_b1") and b2 >= n + (mut == "decide_U2")
                    and (T >= MOD4_BELOW or b3 >= n + (mut == "mod4"))):
                return True, T
        return False, 1 << 20
    if wl + 1 > 256:
        return True, 1 << 20   # too long for the bit-parallel filter: the exact kernel decides
    for k in range(k0, k1 + 1):
        T, _, _, _, _, b1, b2, _ = fb[k]
        if T == 0:
            break
        if b1 >= need(T) and b2 >= need(T) + (mut == "probe_filter_U2"):
            return True, 1 << 20
    return False, 1 << 20


def longest_window(cfg, max_len: int) -> int:
    mode, _, mx, _, _, sl = cfg
    if mode == 2:
        return 2 * sl
    return max_len if max_len < 4 * mx else (max_len + 1) // 2


def unit_filter(cfg, mates: Sequence[bytes], longest: int):
    """(survives, t_hit, kills): whether the restated pipeline keeps the unit, the t_hit of its first passing probe, and the
    mutants under which it would be lost"""
    mode, mn, mx, _, _, sl = cfg
    codes = [encode(m) for m in mates]
    pr = unit_probes(mode, mn, mx, sl, len(mates[0]), len(mates[-1]))

    def run(mut):
        for p in pr:
            ok, t = probe_passes(cfg, codes[p[0]], p, longest, mut)
            if ok:
                return True, t
        return False, 1 << 20
    surv, t_hit = run(None)
    kills = [m for m in MUTANTS if surv and not run(m)[0]]
    return surv, t_hit, kills


# ---------------------------------------------------------------- construction

def _rand(rng: random.Random, n: int) -> bytearray:
    return bytearray(rng.choice(LETTERS) for _ in range(n))


def _unit(rng: random.Random, p: int) -> Tuple[bytearray, int]:
    """a unit of period p with two distinct bases besides one phase (most of its variants are not homopolymers)"""
    while True:
        u = _rand(rng, p)
        j = rng.randrange(p)
        if len(set(u[:j] + u[j + 1:])) >= 2:
            return u, j


def variant_window(rng: random.Random, wl: int, p: int, m_x: int, n_pos: Sequence[int] = ()) -> Optional[bytearray]:
    """wl bases, period p, whose x-class has m_x p-windows (at the start; the other classes after it, each smaller)"""
    u, _ = _unit(rng, p)
    c, j = (m_x - 1) // p + 1, (m_x - 1) % p   # x at phase j of copies 0..c-1: (j + 1) + (c - 1) p windows
    x = rng.choice(LETTERS)
    others = [b for b in LETTERS if b != x]
    rng.shuffle(others)
    ncopy = (wl + p - 1) // p
    rest = ncopy - c
    if rest < 0:
        return None
    w = bytearray()
    for q in range(ncopy):
        v = bytearray(u)
        v[j] = x if q < c else others[min(2, (q - c) * 3 // max(rest, 1))]
        w += v
    w = w[:wl]
    for q in n_pos:
        w[q] = ord("N")
    return w


class Unit:
    __slots__ = ("mates", "margin", "regimes", "kills", "t_hit")

    def __init__(self, mates, margin, regimes, kills=(), t_hit=1 << 20):
        self.mates, self.margin, self.regimes, self.kills, self.t_hit = list(mates), margin, set(regimes), list(kills), t_hit


def _embed(rng: random.Random, cfg, window: bytearray) -> List[bytes]:
    """the read(s) around a probe window: `half` = first half of a short read, `mate1` = segment 1 of a pair, `slice` = the
    whole single-slice long read"""
    mode = cfg[0]
    wl = len(window)
    if mode == 0:
        n = 2 * wl + rng.randint(0, 1)
        return [bytes(window + _rand(rng, n - wl))]
    if mode == 1:
        n1 = 2 * wl + rng.randint(0, 1)
        n2 = rng.choice([n1, n1 - rng.randint(1, 40), n1 + rng.randint(0, 10)])
        return [bytes(window + _rand(rng, n1 - wl)), bytes(_rand(rng, n2))]
    return [bytes(window)]


def _geometry_regimes(cfg, mates, probe, k, T, E, t_hit) -> List[str]:
    mode, mn, mx, low, high, sl = cfg
    _, st, wl, k0, k1 = probe
    clean = all(c in b"ACGT" for c in mates[probe[0]][st:st + wl])
    r = []
    fast = wl <= FAST_MAX_WL and k1 <= 63 and k1 <= wl
    if mode == 2:
        r.append("long_slice")
        if wl > 255:
            r.append("pass_through")
    if mode == 1:
        n = min(len(mates[0]), len(mates[1]))
        r.append("pair_whole" if 4 * mx > n else "pair_segment")
    if fast and clean:
        r.append("screen_fast_E" if E > 0 else "screen_fast")
    elif clean and FAST_MAX_WL < wl <= FAST_MAX_WL_LONG and k1 <= 64:
        r.append("screen_long")
    if fast and not clean:
        r.append("decide_mod4" if T < MOD4_BELOW else "decide_parity")
    if fast and k >= 32:
        r.append("decide_k32")
    if not fast and wl + 1 <= 256:
        r.append("probe_filter5" if wl + 1 <= 160 else "probe_filter8")
    if t_hit in (THREAD_MIN_WINDOWS - 1, THREAD_MIN_WINDOWS, THREAD_MIN_WINDOWS + 1):
        r.append("list_boundary")
    if Oracle.need(T, low) < low * T:
        r.append("need_pre_rounding")
    return r


def margin_pair(o: Oracle, rng: random.Random, cfg, wl: int, p: int, n_count: int, B: float):
    """(read at margin 0, twin at -1, probe, T) against threshold B, or None when the certificate disagrees"""
    n_pos = []
    if n_count:
        lo = min(wl - 1, wl // 2 + 4)
        n_pos = sorted(rng.sample(range(lo, wl), n_count))
    probe_w = bytearray(b"A" * wl)
    for q in n_pos:
        probe_w[q] = ord("N")
    T = sum(1 for i in range(wl - p + 1) if all(probe_w[i + d] != ord("N") for d in range(p)))
    if T <= 0:
        return None
    m_x = Oracle.need(T, B)
    if m_x < 2 or m_x > T:
        return None
    state = rng.getstate()
    out = []
    for m in (m_x, m_x - 1):
        rng.setstate(state)   # the twin differs only in the x-class count
        w = variant_window(rng, wl, p, m, n_pos)
        if w is None:
            return None
        out.append(_embed(rng, cfg, w))
    mode, mn, mx, low, _, sl = cfg
    pr = unit_probes(mode, mn, mx, sl, len(out[0][0]), len(out[0][-1]))
    if unit_margin(o, cfg, out[0], B) != 0 or unit_margin(o, cfg, out[1], B) != -1:
        return None
    if B != low and unit_margin(o, cfg, out[1]) is not None and (unit_margin(o, cfg, out[0]) or -1) < 0:
        return None
    first = pr[0]
    Tk, M, _, _ = o.period_stats(out[0][0], first[1], first[1] + first[2] - 1, p)
    if M != m_x or Tk != T:
        return None
    return out[0], out[1], first, T


def _margin_reads(o: Oracle, rng: random.Random, cfg, name: str, count: int, B: float, tag: str = "") -> List[Unit]:
    """margin-0 reads and their -1 twins in the probe geometries this configuration reaches"""
    mode, mn, mx, low, high, sl = cfg
    units: List[Unit] = []
    tries = 0
    while len(units) < 2 * count and tries < 40 * count:
        tries += 1
        if mode == 2:
            wl = rng.randint(sl, 2 * sl - 1)
            if name.endswith("055") and rng.random() < 0.5:
                wl = rng.randint(128, 131)
            p = rng.randint(mn, mx)
            if name.endswith("055") and wl <= 131:
                p = wl - 99
            n_count = rng.choice([0, 0, 1])
        else:
            shape = rng.random()
            if shape < 0.25:
                wl = rng.randint(50, 64)              # 100..129-base reads
            elif shape < 0.5:
                wl = rng.randint(65, 95)              # E > 0 possible
            elif shape < 0.65:
                wl = rng.randint(96, 159)             # 4-word first level / probe_filter<5>
            else:
                wl = 75
            n = 2 * wl
            k1 = min(n // 4, mx)
            p = rng.randint(mn, k1)
            if rng.random() < 0.3 and k1 >= 32:
                p = rng.randint(32, k1)
            n_count = rng.choice([0, 0, 1, 2])
        got = margin_pair(o, rng, cfg, wl, p, n_count, B)
        if got is None:
            continue
        zero, twin, probe, T = got
        longest = longest_window(cfg, max(len(m) for m in zero))
        for mates, margin in ((zero, 0), (twin, -1)):
            surv, t_hit, kills = unit_filter(cfg, mates, longest)
            E = max(0, T - 64)
            reg = _geometry_regimes(cfg, mates, probe, p, T, E, t_hit)
            if tag:
                reg.append(tag)
            if margin == 0 and rng.random() < 0.5 and mode == 0 and not tag:
                # the same probe window at the end of the half: the x-class windows come last (E > 0 of the first level)
                w = bytearray(mates[0][:probe[2]])[::-1]
                rest = mates[0][probe[2]:]
                rev = [bytes(w) + rest]
                if unit_margin(o, cfg, rev) == 0:
                    s2, t2, k2 = unit_filter(cfg, rev, longest)
                    units.append(Unit(rev, 0, _geometry_regimes(cfg, rev, probe, p, T, E, t2) + ["class_last"], k2, t2))
            units.append(Unit(mates, margin, reg, kills, t_hit))
    return units


# ---------------------------------------------------------------- exact-kernel edges

def _class_counts(seq: bytes, st: int, nd: int, k: int) -> Dict[bytes, int]:
    out: Dict[bytes, int] = {}
    for i in range(st, nd - k + 2):
        w = seq[i:i + k]
        if any(c not in b"ACGT" for c in w):
            continue
        key = min(bytes(w[r:] + w[:r]).translate(bytes.maketrans(b"TGCA", b"0123")) for r in range(k))
        out[key] = out.get(key, 0) + 1
    return out


def ratio_ties(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """a later, non-multiple period p2 whose M/T equals the accepted ratio of p1 (accepted: f >= f_last), and the same read
    with M2 one lower (not accepted); in the first half of a short read"""
    mode, mn, mx, low, high, sl = cfg
    units: List[Unit] = []
    tries = 0
    while len(units) < 2 * count and tries < 400 * count:
        tries += 1
        wl = rng.randint(64, 95)
        p1 = rng.randint(mn, min(wl // 2, mx) // 2)
        p2 = rng.randint(p1 + 1, min(wl // 2, mx))
        if p2 % p1 == 0:
            continue
        T1, T2 = wl - p1 + 1, wl - p2 + 1
        g = math.gcd(T1, T2)
        step = T1 // g
        m1 = step * max(1, math.ceil(Oracle.need(T1, low) / step))
        m2 = m1 * T2 // T1
        L1, L2 = m1 + p1 - 1, m2 + p2 - 1
        gap = wl - L1 - L2
        if gap < 2:
            continue
        u1, u2 = _rand(rng, p1), _rand(rng, p2)
        if len(set(u1)) < 2 or len(set(u2)) < 2:
            continue
        pre = _rand(rng, gap)
        reads = []
        for m in (m2, m2 - 1):
            w = ((u1 * (L1 // p1 + 1))[:L1] + pre + (u2 * ((m + p2 - 1) // p2 + 1))[:m + p2 - 1])
            w += _rand(random.Random(tries), wl - len(w))
            reads.append(bytes(w) + bytes(_rand(random.Random(tries + 1), wl)))
        # certify: equal ratios at p1 and p2, p2 accepted by LOW in the tie read and p1 in the twin
        s = [[o.period_stats(r, 0, wl - 1, k) for k in (p1, p2)] for r in reads]
        (a1, a2), (b1, b2) = s
        if not (a1[1] * a2[0] == a2[1] * a1[0] and b1[1] == a1[1] and b2[1] == a2[1] - 1):
            continue
        tl0 = o.k_mer_check(reads[0], 0, wl - 1, mn, min(len(reads[0]) // 4, mx))[1]
        tl1 = o.k_mer_check(reads[1], 0, wl - 1, mn, min(len(reads[1]) // 4, mx))[1]
        if tl0 != p2 or tl1 != p1:
            continue
        units.append(Unit([reads[0]], unit_margin(o, cfg, [reads[0]]), ["ratio_tie"]))
        units.append(Unit([reads[1]], unit_margin(o, cfg, [reads[1]]), ["ratio_below"]))
    return units


def homopolymer_ties(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """a poly-A run and a repeat whose classes tie at period p, in both orders: cls_max takes the class that reaches the
    maximum first, so p is accepted only when the repeat comes first"""
    mode, mn, mx, low, high, sl = cfg
    units: List[Unit] = []
    tries = 0
    while len(units) < 2 * count and tries < 400 * count:
        tries += 1
        wl = rng.randint(64, 95)
        p = rng.randint(mn, min(12, mx))
        L = rng.randint(Oracle.need(wl - p + 1, low) + p - 1, (wl - 2) // 2)
        u = _rand(rng, p)
        if b"A" in u or len(set(u)) < 2:
            continue
        rep, hom, gap = (u * (L // p + 1))[:L], b"A" * L, _rand(rng, wl - 2 * L)
        if b"A" in gap:
            gap = gap.replace(b"A", b"C")
        tail = bytes(_rand(rng, wl))
        pair = [bytes(rep + gap + hom) + tail, bytes(hom + gap + rep) + tail]
        ok = True
        tls = []
        for r in pair:
            cc = _class_counts(r, 0, wl - 1, p)
            top = sorted(cc.values(), reverse=True)
            if len(top) < 2 or top[0] != top[1] or top[0] < Oracle.need(wl - p + 1, low):
                ok = False
                break
            tls.append(o.k_mer_check(r, 0, wl - 1, mn, min(len(r) // 4, mx))[1])
        if not ok or tls[0] != p or tls[1] == p:
            continue
        units.append(Unit([pair[0]], unit_margin(o, cfg, [pair[0]]), ["homopolymer_tie"]))
        units.append(Unit([pair[1]], unit_margin(o, cfg, [pair[1]]), ["homopolymer_tie"]))
    return units


def divisor_reads(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """periods p and 2p both at margin >= 0 (2p is blocked by its accepted divisor)"""
    mode, mn, mx, low, high, sl = cfg
    units: List[Unit] = []
    tries = 0
    while len(units) < count and tries < 100 * count:
        tries += 1
        wl = rng.randint(60, 80)
        p = rng.randint(mn, min(wl // 2, mx) // 2)
        u = _rand(rng, p)
        if len(set(u)) < 2:
            continue
        L = rng.randint(int(0.85 * wl), wl)
        w = (u * (wl // p + 1))[:L] + _rand(rng, wl - L)
        r = bytes(w) + bytes(_rand(rng, wl))
        ok = True
        for k in (p, 2 * p):
            T, M, _, _ = o.period_stats(r, 0, wl - 1, k)
            ok = ok and T > 0 and M >= Oracle.need(T, low)
        if ok and o.k_mer_check(r, 0, wl - 1, mn, min(len(r) // 4, mx))[1] == p:
            units.append(Unit([r], unit_margin(o, cfg, [r]), ["divisor"]))
    return units


def high_edges(o: Oracle, rng: random.Random, cfg, count: int) -> List[Unit]:
    """margin 0 against HIGH (target_k_high) as well"""
    units = _margin_reads(o, rng, cfg, "", count, cfg[4], tag="high_edge")
    for u in units:   # the margin against HIGH is 0 or -1; what is recorded is the margin against LOW
        if u.margin == -1:
            u.regimes = {r for r in u.regimes if r != "high_edge"} | {"high_edge_twin"}
        u.margin = unit_margin(o, cfg, u.mates)
    return units


def corpus(name: str, seed: int = 1, count: int = 40) -> List[Unit]:
    """the edge corpus of one configuration"""
    cfg = CONFIGS[name]
    mode, mn, mx, low, high, sl = cfg
    o = Oracle(mn, mx, low, high, slice_len=sl)
    rng = random.Random(seed * 1000003 + sum(map(ord, name)))
    units = _margin_reads(o, rng, cfg, name, count, low)
    if mode == 0:
        units += divisor_reads(o, rng, cfg, count // 4)
        if high < 1.0 and high != low:
            units += high_edges(o, rng, cfg, count // 4)
        if low <= 0.45:
            units += ratio_ties(o, rng, cfg, count // 4)
            units += homopolymer_ties(o, rng, cfg, count // 4)
    return units


def regime_counts(units: Sequence[Unit]) -> Dict[str, Tuple[int, int, int]]:
    """regime -> (reads at margin 0, reads at margin -1, all reads)"""
    out: Dict[str, List[int]] = {}
    for u in units:
        for r in u.regimes:
            c = out.setdefault(r, [0, 0, 0])
            c[0] += u.margin == 0
            c[1] += u.margin == -1
            c[2] += 1
    return {k: (v[0], v[1], v[2]) for k, v in sorted(out.items())}


def kill_counts(units: Sequence[Unit]) -> Dict[str, int]:
    out = {m: 0 for m in MUTANTS}
    for u in units:
        for m in u.kills:
            out[m] += 1
    return out


def scan_args(name: str, units: Sequence[Unit]):
    """(mode, reads1, reads2) for Oracle.scan / DeviceContext.submit_reads"""
    mode = CONFIGS[name][0]
    r1 = [u.mates[0] for u in units]
    r2 = [u.mates[1] for u in units] if mode == 1 else None
    return mode, r1, r2
