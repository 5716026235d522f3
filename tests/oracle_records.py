"""Per-unit records from the CPU oracle, for the unit-record tests.  TEST INFRASTRUCTURE ONLY.

A unit (a read; a pair in paired mode) leaves nothing behind for the next one in the oracle's routing: the temp maps are
empty again when it is done (the pair-leak emulation aside, which records are not defined for).  So a unit's records --
its adds into the six final maps, adds to the same key merged -- are the tables of a scan of that unit alone."""
from typing import Dict, Optional, Sequence, Tuple

UnitRecords = Dict[Tuple[int, int, int, int], int]   # (unit, table, k, seq) -> count


def scan_records(oracle, mode: int, reads1: Sequence[bytes], reads2: Optional[Sequence[bytes]] = None) -> UnitRecords:
    """{(unit, table, k, seq): count}; unit = the 0-based index of the read (of the pair in mode 1, pairs matched
    index-wise up to the shorter list)."""
    assert not oracle.cfg.emulate_pair_leak, "unit records are defined without the pair leak emulation"
    n = min(len(reads1), len(reads2 or [])) if mode == 1 else len(reads1)
    out: UnitRecords = {}
    for u in range(n):
        tables = oracle.scan(mode, [reads1[u]], [reads2[u]] if mode == 1 else None)
        for (tb, k, s), c in tables.items():
            out[(u, tb, k, s)] = c
    return out
