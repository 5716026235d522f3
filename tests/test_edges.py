"""Reads on an acceptance threshold (oracle/edges.py), checked without a GPU: the generator's certificates and coverage,
the oracle's per-period statistics, and the host build of the thread-per-read exact kernels (exact_thread.cuh) on the
corpus -- ratio ties, homopolymer ties, blocked divisors and windows whose best period sits exactly on need(T)."""
import random

import pytest

from oracle import edges
from oracle.oracle import Oracle
from trew_b200 import synth

from test_exact_thread import etc, run, run_pairs   # noqa: F401  (etc is a fixture)

# regime -> the fewest reads at margin 0 (and as many twins at -1) each configuration of that mode must hold
MIN_SHORT = {"screen_fast": 4, "screen_fast_E": 1, "screen_long": 1, "probe_filter5": 2, "class_last": 4}
MIN_PAIR = {"pair_segment": 1, "pair_whole": 4, "screen_fast": 4, "probe_filter5": 2}
MIN_LONG = {"long_slice": 20, "probe_filter8": 8}
# regime -> the fewest reads of it over all configurations, whatever their margin
MIN_ANY = {"decide_mod4": 20, "decide_parity": 10, "decide_k32": 10, "pass_through": 4, "list_boundary": 3, "need_pre_rounding": 8,
           "ratio_tie": 4, "ratio_below": 4, "homopolymer_tie": 4, "divisor": 20, "high_edge": 10, "high_edge_twin": 10}
# mutant -> the fewest units of the whole corpus it would lose (the restated filter pipeline says so)
MIN_KILLS = {"fast_entry": 30, "decide_E": 60, "decide_b1": 60, "decide_U2": 60, "mod4": 30, "probe_filter_U2": 30}


@pytest.fixture(scope="module")
def corpora():
    return {name: edges.corpus(name) for name in edges.CONFIGS}


def test_period_stats_rebuild_select_k(kmer_check_cases):
    """select_k restated from Oracle.period_stats gives k_mer_check's (th, tl): on the reference's golden cases and on
    adversarial windows"""
    def select(o, seq, st, nd, kmin, kmax, B):
        tk, tf, acc = 0, 0.0, []
        for k in range(kmin, kmax + 1):
            T, M, S, _ = o.period_stats(seq, st, nd, k)
            if T == 0:
                continue
            f = M / T
            if f >= max(B, tf) and not o.homo(S, k) and not any(k % a == 0 for a in acc):
                tk, tf = k, f
                acc.append(k)
        return tk
    cases = [(c["min_mer"], c["max_mer"], c["seq"].encode(), c["st"], c["nd"], c["kmin"], c["kmax"]) for c in kmer_check_cases]
    rng = random.Random(5)
    for r in synth.adversarial_short(31, 300, max_unit=40):
        if len(r) >= 20:
            cases.append((5, 40, r, 0, len(r) // 2 - 1, 5, min(len(r) // 4, 40)))
    assert len(cases) > 300
    for mn, mx, seq, st, nd, kmin, kmax in cases:
        o = Oracle(mn, mx, rng.choice([0.5, 0.35]), 0.8)
        th, tl = o.k_mer_check(seq, st, nd, kmin, kmax)[:2]
        assert (th, tl) == (select(o, seq, st, nd, kmin, kmax, o.cfg.high), select(o, seq, st, nd, kmin, kmax, o.cfg.low))
    assert [Oracle.need(T, 0.5) for T in (1, 2, 3, 10)] == [1, 1, 2, 5] and Oracle.need(100, 0.55) == 55 and Oracle.need(7, 1.1) == 8


def test_generator_is_certified_and_covers_every_regime(corpora):
    """Every read's margin is what the generator says, each regime holds its minimum of margin-0 reads and -1 twins, and
    the corpus holds reads that a one-tighter comparison in each filter level would lose.  Run with -s for the counts."""
    total, kills = {}, {m: 0 for m in edges.MUTANTS}
    for name, units in corpora.items():
        cfg = edges.CONFIGS[name]
        o = Oracle(*cfg[1:5], slice_len=cfg[5])
        counts = edges.regime_counts(units)
        print("\n%-14s %4d units  %s" % (name, len(units), "  ".join("%s %d/%d/%d" % (r, *c) for r, c in counts.items())))
        mins = (MIN_SHORT, MIN_PAIR, MIN_LONG)[cfg[0]]
        for r, n in mins.items():
            assert counts.get(r, (0, 0, 0))[0] >= n, (name, r, counts.get(r))
            if r != "class_last":
                assert counts[r][1] >= n, (name, r, counts[r])
        for r, c in counts.items():
            total[r] = total.get(r, 0) + c[2]
        for u in units:
            assert edges.unit_margin(o, cfg, u.mates) == u.margin   # re-certified from scratch
            # the restated filters are sound: a unit some probe of which reaches LOW survives them
            surv, _, k = edges.unit_filter(cfg, u.mates, edges.longest_window(cfg, max(len(r) for u2 in units for r in u2.mates)))
            assert surv or u.margin is None or u.margin < 0
            for m in u.kills:
                kills[m] += 1
    print("regimes over all configurations:", total)
    print("units each one-tighter comparison would lose:", kills)
    for r, n in MIN_ANY.items():
        assert total.get(r, 0) >= n, (r, total.get(r))
    for m, n in MIN_KILLS.items():
        assert kills[m] >= n, (m, kills[m])


def test_generator_is_deterministic():
    a, b = edges.corpus("short_5_32", seed=3, count=6), edges.corpus("short_5_32", seed=3, count=6)
    assert [u.mates for u in a] == [u.mates for u in b] and len(a) >= 12


@pytest.mark.parametrize("name", [n for n, c in edges.CONFIGS.items() if c[0] == 0])
def test_thread_kernel_on_edges(etc, name):   # noqa: F811
    """exact_thread.cuh on the host, 64- and 128-bit keys, bit-exact against the oracle on the edge corpus"""
    _, mn, mx, low, high, sl = edges.CONFIGS[name]
    units = edges.corpus(name)
    reads = [u.mates[0] for u in units]
    want_all = Oracle(mn, mx, low, high).scan(0, reads)
    assert want_all
    for wide in ([False, True] if mx <= 32 else [True]):
        got, bailed = run(etc, reads, mn, mx, low, high, wide=wide)
        keep = [r for i, r in enumerate(reads) if i not in set(bailed)]
        want = want_all if not bailed else Oracle(mn, mx, low, high).scan(0, keep)
        assert bailed == [i for i, r in enumerate(reads) if len(r) > 160]
        assert got == want, (name, wide, sorted(set(got.items()) ^ set(want.items()))[:6])
        # each exact-kernel edge on its own, so that a failure names it
        for regime in ("ratio_tie", "ratio_below", "homopolymer_tie", "divisor", "high_edge", "high_edge_twin"):
            sub = [u.mates[0] for u in units if regime in u.regimes and len(u.mates[0]) <= 160]
            if sub:
                assert run(etc, sub, mn, mx, low, high, wide=wide)[0] == Oracle(mn, mx, low, high).scan(0, sub), (name, regime, wide)


@pytest.mark.parametrize("name", [n for n, c in edges.CONFIGS.items() if c[0] == 1 and 4 * c[2] <= 150])
def test_thread_pair_kernel_on_edges(etc, name):   # noqa: F811
    """pairs whose shorter mate is below 4 * MAX_MER are outside the thread kernel's limits (the warp kernel takes them)"""
    _, mn, mx, low, high, sl = edges.CONFIGS[name]
    units = edges.corpus(name)
    r1, r2 = [u.mates[0] for u in units], [u.mates[1] for u in units]
    for wide in ([False, True] if mx <= 32 else [True]):
        got, bailed = run_pairs(etc, r1, r2, mn, mx, low, high, wide=wide)
        skip = set(bailed)
        want = Oracle(mn, mx, low, high).scan(1, [r for i, r in enumerate(r1) if i not in skip], [r for i, r in enumerate(r2) if i not in skip])
        assert len(skip) < len(units) and got == want, (name, wide, sorted(set(got.items()) ^ set(want.items()))[:6])
