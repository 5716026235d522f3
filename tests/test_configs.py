"""The configuration grid (oracle/configs.py), checked without a GPU: the grid stays inside what the command line accepts,
every corpus is deterministic and holds its minimum of units per regime, every certificate holds again from scratch, and
the host build of the thread-per-read exact routing (exact_thread.cuh) equals the oracle on every configuration it
supports -- short, paired and long, 64- and 128-bit -- bailing out exactly where test_exact_thread.py says it does."""
import pytest

from oracle import configs as cf
from oracle import edges
from test_exact_thread import etc, run, run_long, run_pairs   # noqa: F401  (etc: the host build, a module fixture)

NAMES = list(cf.CONFIGS)


@pytest.fixture(scope="module")
def corpora():
    return {name: cf.corpus(name) for name in NAMES}


def test_grid_is_inside_the_accepted_range():
    for name, (mode, mn, mx, low, high, sl) in cf.CONFIGS.items():
        assert mode in (0, 1, 2) and 3 <= mn <= mx <= 64 and 0 < low <= high <= 1, name
        assert mode != 2 or 2 * mx <= sl <= 512, name
    values = list(cf.CONFIGS.values())
    for mx in cf.BOUNDARY_MAX:   # each boundary MAX_MER with MIN_MER 3, MIN_MER = MAX_MER and one in between
        mins = {c[1] for c in values if c[0] == 0 and c[2] == mx and (c[3], c[4]) == (0.5, 0.8)}
        assert {3, mx} <= mins and (len(mins) >= 3 or mx <= 4), (mx, mins)
    for mode in (0, 1):
        lows = {(c[3], c[4]) for c in values if c[0] == mode}
        assert set(cf.BASELINES) <= lows and {(b, b) for b in cf.NEXT_ABOVE} <= lows, mode
    slices = {(c[2], c[5]) for c in values if c[0] == 2}
    assert {(3, 6), (5, 10), (20, 40), (32, 64), (64, 128), (64, 512)} <= slices
    assert {s for m, s in slices if m == 32} >= {79, 80, 128, 129, 159, 160} and {(23, 47), (23, 48)} <= slices
    assert sum(name.startswith("random_") for name in NAMES) == 20


def test_corpus_is_deterministic():
    for name in ("short_3_64", "pair_5_32_0.050000000000000003_0.10000000000000001", "long_3_3_s6", "random_05"):
        a, b = cf.corpus(name, seed=2), cf.corpus(name, seed=2)
        assert [u.mates for u in a] == [u.mates for u in b] and [u.regimes for u in a] == [u.regimes for u in b]
        assert [u.mates for u in a] != [u.mates for u in cf.corpus(name, seed=3)]


def test_every_configuration_holds_its_regimes(corpora):
    for name, units in corpora.items():
        counts = cf.regime_counts(units)
        for regime, least in cf.expected_regimes(name).items():
            assert counts.get(regime, 0) >= least, (name, regime, counts.get(regime, 0), least)
        mode = cf.CONFIGS[name][0]
        for u in units:
            assert cf._fits(cf.CONFIGS[name], u.mates) and len(u.mates) == (2 if mode == 1 else 1), name
    tags = lambda name: set().union(*(u.regimes for u in corpora[name]))
    # the branches of the geometry table, seen from the branch tags
    for name in ("short_3_64", "short_40_41", "short_19_37"):
        assert {"thread", "warp", "whole_read_probe", "probe_filter3", "probe_filter5"} <= tags(name), name
    assert "probe_filter8" in tags("short_3_64") and "probe_filter8" in tags("short_40_41")   # whole reads of 255 / 163 bases
    for name in ("pair_3_41", "pair_40_41"):
        assert {"thread", "warp", "unequal_mates", "whole_read_probe"} <= tags(name), name
    for sl in (47, 48, 79, 80, 128, 129, 159, 160):
        t = tags("long_5_%d_s%d" % (23 if sl < 64 else 32, sl))
        assert {"slice_dropped", "single_slice", "multi_slice"} <= t and ("screen_skipped" in t) == (sl >= 160), sl
        assert ("probe_filter8" in t) == (sl > 80) and ("pass_through" in t) == (sl >= 129), sl   # windows of SL .. 2 SL - 1
    assert "hundreds_of_slices" in tags("long_3_3_s6") and "hundreds_of_slices" in tags("long_3_5_s10")
    dense = [n for n in NAMES if cf.CONFIGS[n][3] <= cf.DENSE_LOW and cf.CONFIGS[n][0] == 0]
    assert len(dense) >= 5 and all("dense" in tags(n) for n in dense)


def test_certificates_hold_from_scratch(corpora):
    for name, units in corpora.items():
        cfg = cf.CONFIGS[name]
        o = cf.oracle_for(cfg)
        for u in units:
            assert cf.certify(o, cfg, u) == [], (name, sorted(u.regimes))
        # margin twins: one unit at 0 for each at -1, against the same baseline
        for side in ("low", "high"):
            assert cf.regime_counts(units).get("margin_%s_0" % side) == cf.regime_counts(units).get("margin_%s_-1" % side), name


def test_whole64_is_the_only_accepted_period():
    """the k = 64 unit the screen's fast_span_long<2> alone sees: at MAX_MER 64 a 128..159-base read, periods 3..63 of
    every probe below LOW, 64 accepted in the whole-read probe"""
    for name in ("short_3_64", "short_40_64", "pair_64_64"):
        cfg = cf.CONFIGS[name]
        units = [u for u in cf.corpus(name) if "whole64" in u.regimes]
        assert len(units) >= 3, name
        for u in units:
            pr = edges.unit_probes(cfg[0], cfg[1], cfg[2], cfg[5], len(u.mates[0]), len(u.mates[-1]))
            assert any(p[1] == 0 and p[2] == len(u.mates[0]) and p[4] == 64 for p in pr)
            assert 128 <= len(u.mates[0]) <= 159


@pytest.mark.parametrize("name", NAMES)
def test_host_thread_path_equals_oracle(etc, corpora, name):   # noqa: F811
    mode, mn, mx, low, high, sl = cf.CONFIGS[name]
    units = corpora[name]
    o = cf.oracle_for(cf.CONFIGS[name])
    _, r1, r2 = cf.scan_args(name, units)
    wide = mx > 32
    if mode == 0:
        got, bailed = run(etc, r1, mn, mx, low, high, wide=wide)
        assert bailed == [i for i, r in enumerate(r1) if len(r) > 160 and len(r) >= 2 * mn]
        keep = [r for i, r in enumerate(r1) if i not in set(bailed)]
        want = o.scan(0, keep)
    elif mode == 1:
        got, bailed = run_pairs(etc, r1, r2, mn, mx, low, high, wide=wide)
        assert bailed == [i for i, (a, b) in enumerate(zip(r1, r2))
                          if min(len(a), len(b)) >= 2 * mn and (max(len(a), len(b)) > 160 or min(len(a), len(b)) < 4 * mx)]
        skip = set(bailed)
        want = o.scan(1, [r for i, r in enumerate(r1) if i not in skip], [r for i, r in enumerate(r2) if i not in skip])
    else:
        if mx > 32 or sl > 160:
            pytest.skip("the thread path's long-read steps take MAX_MER <= 32 and SLICE <= 160")
        got, bailed = run_long(etc, r1, mn, mx, sl, low, high)
        keep = [r for i, r in enumerate(r1) if i not in set(bailed)]
        want = o.scan(2, keep)
        assert len(bailed) < len(r1)
    assert got == want, (name, len(got), len(want), sorted(set(got.items()) ^ set(want.items()))[:6])
    assert got or (mode == 1 and 4 * mx > 160), name   # there every pair the thread path could take is below 2 MIN_MER
