"""The CUDA scan on reads that sit exactly on an acceptance threshold (oracle/edges.py): tables per configuration and
regime, the filters' soundness counted directly (every unit a probe of which reaches LOW is a survivor), and both exact
kernels on the whole corpus through the routing switches.

TREW_THREAD_MIN_WINDOWS and TREW_MOD4_BELOW are read once per process, so those runs happen in a child process: this
file run as a script scans every corpus and prints the tables as JSON."""
import json
import os
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import edges   # noqa: E402
from oracle.oracle import Oracle   # noqa: E402
from trew_b200 import api   # noqa: E402

pytestmark = pytest.mark.gpu

NAMES = list(edges.CONFIGS)


def scan(name, units):
    mode, mn, mx, low, high, sl = edges.CONFIGS[name]
    _, r1, r2 = edges.scan_args(name, units)
    with api.DeviceContext(mode, mn, mx, low, high, sl) as ctx:
        ctx.submit_reads(r1, r2)
        return ctx.finish(), ctx.stats().survivors


def oracle_tables(name, units):
    mode, mn, mx, low, high, sl = edges.CONFIGS[name]
    _, r1, r2 = edges.scan_args(name, units)
    return Oracle(mn, mx, low, high, slice_len=sl).scan(mode, r1, r2)


@pytest.fixture(scope="module")
def corpora():
    t = time.time()
    c = {name: edges.corpus(name) for name in NAMES}
    want = {name: oracle_tables(name, c[name]) for name in NAMES}
    print("\nedge corpora: %d units, generated and scanned by the oracle in %.1f s" % (sum(map(len, c.values())), time.time() - t))
    return c, want


def test_tables_per_regime(corpora):
    c, want = corpora
    for name in NAMES:
        got, _ = scan(name, c[name])
        assert got == want[name], name
        for regime in sorted({r for u in c[name] for r in u.regimes}):
            sub = [u for u in c[name] if regime in u.regimes]
            assert scan(name, sub)[0] == oracle_tables(name, sub), (name, regime)


def test_must_survive_units_are_survivors(corpora):
    """stats().survivors counts list A plus list B (disjoint): one unit lost by a filter shows as one short, even when it
    would have emitted nothing"""
    c, _ = corpora
    for name in NAMES:
        must = [u for u in c[name] if u.margin is not None and u.margin >= 0]
        assert len(must) > 10
        _, surv = scan(name, must)
        assert surv == len(must), (name, surv, len(must))
        _, surv_all = scan(name, c[name])
        assert surv_all >= len(must), (name, surv_all, len(must))


@pytest.mark.parametrize("flags", ["4", "1", "2", "5", "6"])
def test_exact_flags_routings(corpora, monkeypatch, flags):
    """4: the warp kernel for every survivor; 1: its serial eval_k path; 2: without the composition bound"""
    c, want = corpora
    monkeypatch.setenv("TREW_EXACT_FLAGS", flags)
    for name in NAMES:
        assert scan(name, c[name])[0] == want[name], (name, flags)


def child_tables(env):
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=dict(os.environ, **env), capture_output=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.decode().strip().splitlines()[-1])
    return {name: ({(t, k, s): n for t, k, s, n in rows}, surv) for name, (rows, surv) in out.items()}


@pytest.mark.parametrize("env", [{"TREW_THREAD_MIN_WINDOWS": "0"}, {"TREW_MOD4_BELOW": "0"}, {"TREW_MOD4_BELOW": "100000"}],
                         ids=["thread_min_windows_0", "mod4_off", "mod4_always"])
def test_process_wide_switches(corpora, env):
    """TREW_THREAD_MIN_WINDOWS=0 puts every survivor of up to 160 bases through the thread kernel; TREW_MOD4_BELOW=0 turns the
    decide kernel's third level off, 100000 asks it for every period.  The third level may only remove survivors."""
    c, want = corpora
    got = child_tables(env)
    for name in NAMES:
        assert got[name][0] == want[name], (name, env)
    if env.get("TREW_MOD4_BELOW") == "0":
        base = {name: scan(name, c[name])[1] for name in NAMES}
        assert all(base[name] <= got[name][1] for name in NAMES), (base, {n: g[1] for n, g in got.items()})


if __name__ == "__main__":
    res = {}
    for name in NAMES:
        tables, surv = scan(name, edges.corpus(name))
        res[name] = ([[t, k, s, n] for (t, k, s), n in sorted(tables.items())], surv)
    print(json.dumps(res))
