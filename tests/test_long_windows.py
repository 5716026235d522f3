"""Windows of 161 up to 1023 bases (oracle/long_windows.py), checked without a GPU: the corpus is deterministic, holds every
length of its table in every configuration, and every constructed regime holds its minimum of units, each one certified
again from scratch with the oracle's per-period statistics.  Also the host-side check of packed batches
(trew_check_batch) on hand-built trew_batch structs."""
import ctypes as C

import numpy as np
import pytest

from oracle import edges
from oracle import long_windows as lw
from oracle.oracle import Oracle
from trew_b200 import api

# regime -> configurations that must hold at least this many units of it
MIN_REGIME = {
    "limit_10bit": ({"pair_5_32", "pair_3_64", "long_5_32_s512", "long_3_64_s512"}, 3),
    "many_classes": ({"long_5_32_s512", "long_3_64_s512"}, 2),
    "few_windows": ({"long_5_32_s512", "long_3_64_s512"}, 3),
    "few_runs": ({"short_5_32", "pair_5_32", "pair_3_64", "long_5_32_s512", "long_3_64_s512", "long_5_32_s300"}, 3),
    "margin_edge": ({"short_5_32", "pair_5_32", "pair_3_64", "long_5_32_s512"}, 8),
}


@pytest.fixture(scope="module")
def corpora():
    return {name: lw.corpus(name) for name in lw.CONFIGS}


def test_corpus_is_deterministic():
    for name in ("short_3_64", "pair_3_64", "long_5_32_s512"):
        a, b = lw.corpus(name, seed=2), lw.corpus(name, seed=2)
        assert [u.mates for u in a] == [u.mates for u in b] and [u.regimes for u in a] == [u.regimes for u in b]
        assert [u.mates for u in a] != [u.mates for u in lw.corpus(name, seed=3)]


def test_every_length_in_every_configuration(corpora):
    for name, units in corpora.items():
        mode, mn, mx, _, _, sl = lw.CONFIGS[name]
        keys = {u.length for u in units}
        assert set(lw.lengths(name)) <= keys, (name, set(lw.lengths(name)) - keys)
        for u in units:
            n1, n2 = len(u.mates[0]), len(u.mates[-1])
            if isinstance(u.length, int) and not u.regimes & set(lw.REGIMES):
                assert n1 == u.length, (name, u.length, n1)
            elif isinstance(u.length, tuple) and u.length[0] == "trunc":
                assert n1 == u.length[1] and 1 <= n2 <= n1
            elif isinstance(u.length, tuple):
                assert (n1, n2) == u.length
            elif u.length == "4-20kb":
                assert 4000 <= n1 <= 20000
            elif u.length == "50-200kb":
                assert 50000 <= n1 <= 200000 and "hundreds_of_slices" in u.regimes
            # every unit stays inside what submit_chunk accepts
            assert max(n1, n2) <= (1000 if mode == 0 else 1023 if mode == 1 else 1 << 20)
    # the table's boundaries, seen from the geometry tags
    tags = lambda name: set().union(*(u.regimes for u in corpora[name]))
    for name in ("short_5_32", "short_3_64", "short_12_40", "short_035_06"):
        assert {"thread", "warp", "whole_read_probe", "probe_filter5", "probe_filter8", "pass_through"} <= tags(name), name
    assert "probe_filter8" in tags("short_3_64") and "pass_through" in tags("short_3_64")   # 255 / 256: the whole read at 3 64
    for name in ("pair_5_32", "pair_3_64", "pair_12_40"):
        assert {"warp", "truncated_mate", "unequal_mates", "window_512_plus"} <= tags(name), name
    assert "window_1023" in tags("pair_3_64") and "window_1023" in tags("long_5_32_s512") and "window_1023" in tags("long_3_64_s512")
    for sl in lw.SLICES:
        t = tags("long_5_32_s%d" % sl)
        assert {"slice_dropped", "single_slice", "multi_slice"} <= t, sl
        assert ("screen_skipped" in t) == (sl > 159) and ("slice_over_160" in t) == (sl > 80)
    assert "hundreds_of_slices" in tags("long_5_32_s64") and "hundreds_of_slices" in tags("long_3_64_s128")


def _first_probe(cfg, mates):
    mode, mn, mx, _, _, sl = cfg
    return edges.unit_probes(mode, mn, mx, sl, len(mates[0]), len(mates[-1]))[0]


def test_regimes_hold_their_minimum_and_certify(corpora):
    """each constructed unit re-certified: the statistics its regime is named for hold at the window the kernel scans"""
    for regime, (names, least) in MIN_REGIME.items():
        for name in names:
            cfg = lw.CONFIGS[name]
            mode, mn, mx, low, high, sl = cfg
            o = Oracle(mn, mx, low, high, slice_len=sl)
            units = [u for u in corpora[name] if regime in u.regimes]
            assert len(units) >= least, (name, regime, len(units))
            for u in units:
                m = u.mates[0]
                _, st, wl, k0, k1 = _first_probe(cfg, u.mates)
                nd = st + wl - 1
                if regime == "limit_10bit":
                    assert wl == 1023 and k0 == mn and o.period_stats(m, st, nd, mn)[:2] == (1024 - mn, 1024 - mn)
                elif regime == "many_classes":
                    th, tl = o.k_mer_check(m, st, nd, k0, k1)[:2]
                    k = tl or th
                    assert wl == 1023 and k and o.period_stats(m, st, nd, k)[3] >= 300
                    assert lw.match_runs(m, st, nd, k) > lw.SERIAL_MAX_RUNS
                elif regime == "few_windows":
                    few = [k for k in range(k0, k1 + 1) if 0 < o.period_stats(m, st, nd, k)[0] <= 32]
                    assert wl == 1023 and few, name
                    k = few[-1]
                    lanes = {i // 32 for i in range(wl - k + 1) if b"N" not in m[st + i:st + i + k]}
                    assert len(lanes) >= 12
                elif regime == "few_runs":
                    tl = o.k_mer_check(m, st, nd, k0, k1)[1]
                    assert wl >= 500 and tl and lw.match_runs(m, st, nd, tl) <= lw.SERIAL_MAX_RUNS
                elif regime == "margin_edge":
                    assert edges.unit_margin(o, cfg, u.mates) in (0, -1)
            if regime == "margin_edge":
                margins = [edges.unit_margin(o, cfg, u.mates) for u in units]
                assert margins.count(0) == margins.count(-1) >= least // 2
                assert {u.length for u in units} == {w for w in lw.MARGIN_WINDOWS[mode] if mode != 2 or sl <= w < 2 * sl}


def test_match_runs():
    assert lw.match_runs(b"ACG" * 50, 0, 149, 3) == 1
    assert lw.match_runs(b"ACGT" * 10 + b"N" + b"ACGT" * 10, 0, 80, 4) == 2
    r = bytearray(b"ACG" * 50)
    r[70] = ord("T")   # windows 67..70 leave the run; 71 on start a new one
    assert lw.match_runs(bytes(r), 0, 149, 3) == 3


# ---- trew_check_batch ------------------------------------------------------------------------------------------------------

def check(mode, lens=None, max_read_len=None, bit_off=None, n_reads=None):
    L = api.load_library()
    off = np.array(bit_off if bit_off is not None else np.concatenate([[0], np.cumsum(lens)]), dtype=np.uint32)
    b = api.Batch()
    b.n_reads = len(off) - 1 if n_reads is None else n_reads
    b.max_read_len = max(lens) if max_read_len is None else max_read_len
    b.bit_off = off.ctypes.data_as(C.POINTER(C.c_uint32))   # the check reads bit_off only
    return L.trew_check_batch(mode, C.byref(b))


S, P, LONG = api.MODE_SHORT, api.MODE_PAIR, api.MODE_LONG


def test_check_batch_accepts_what_the_packers_make():
    assert check(S, [150, 1000, 3]) == 0
    assert check(S, [150, 200], max_read_len=5000) == 0    # larger than the longest read: a larger workspace, allowed
    assert check(P, [1023, 40, 150, 150]) == 0
    assert check(LONG, [200000, 64]) == 0                  # long mode has no length limit
    assert check(S, [], max_read_len=0, bit_off=[0]) == 0  # an empty batch
    reads = [b"ACGT" * 50, b"TTAGGG" * 166, b"A" * 7]
    buf, locs = api.make_chunk(reads)
    pb = api.PackedBatch(buf, locs)
    assert pb.batch.max_read_len == 996 and api.load_library().trew_check_batch(S, C.byref(pb.batch)) == 0
    pp = api.PackedBatch(buf, locs, n_ranges=1, buf2=buf, locs2=locs)
    assert pp.batch.max_read_len == 996 and api.load_library().trew_check_batch(P, C.byref(pp.batch)) == 0


def test_check_batch_rejects_an_understated_max_read_len():
    assert check(S, [150, 200], max_read_len=199) == 1
    assert check(P, [1023, 40], max_read_len=1022) == 1
    assert check(LONG, [20000, 3000], max_read_len=19999) == 1
    assert check(LONG, [20000, 3000], max_read_len=0) == 1


def test_check_batch_rejects_bad_offsets():
    assert check(S, [10], bit_off=[4, 14]) == 1            # bit_off[0] != 0
    assert check(S, [10, 10], bit_off=[0, 20, 10]) == 1    # decreasing
    assert check(LONG, [10, 10], bit_off=[0, 10, 10, 5], max_read_len=10) == 1
    assert check(S, [10], bit_off=[0, 10, 10], max_read_len=10) == 0   # a read of 0 bases is fine


def test_check_batch_rejects_an_odd_pair_batch():
    assert check(P, [150, 150, 150]) == 1
    assert check(S, [150, 150, 150]) == 0


def test_check_batch_length_limits_match_submit_chunk():
    assert check(S, [1000, 20]) == 0
    assert check(S, [20, 1001]) == 4                       # TREW_ERR_TOO_LONG, as submit_chunk gives it
    assert check(S, [20, 1023]) == 4
    assert check(P, [1023, 1023]) == 0
    assert check(P, [150, 1024]) == 4
    assert check(P, [5000, 150]) == 4
    assert check(7, [150]) == 1                            # no such mode
    assert api.load_library().trew_check_batch(S, None) == 1
