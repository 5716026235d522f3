"""ctypes front-ends for the two CPU checkers.  TEST INFRASTRUCTURE ONLY.

* ``Oracle``     -- oracle/trew_oracle.c, the plain-C restatement (always available; built by
                    ``make -C oracle`` / ``__graft_entry__.build()`` into oracle/_build/).
* ``Reference``  -- oracle/_ref/libtrew_ref.so, the UNMODIFIED reference src/kmer.cpp compiled
                    against shim headers (only where it was built, i.e. where /root/reference
                    existed at build time; the prebuilt .so travels to the GPU box).

Only tests/, tools/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module.  The product package (trew_b200) must not.

Both classes expose the same interface so tests can diff them:

    scan(mode, reads1, reads2=None) -> {(table, k, seq): count}
        mode 0 short single-end (buffer_task, src/kmer.cpp:80), 1 paired (buffer_task_pair, :268),
        2 long (buffer_task_long, :747).  table ids: 0 F_h 1 F_l 2 B_h 3 B_l 4 O_h 5 O_l.
    k_mer_check(seq, st, nd, kmin, kmax) -> (th, tl, S_h, S_l, {(cls, k, seq): count})
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "_build", "libtrew_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libtrew_ref.so")
REF_BIN = os.path.join(HERE, "_ref", "trew_ref")

TABLE_NAMES = ("F_h", "F_l", "B_h", "B_l", "O_h", "O_l")
LETTERS = "TGCA"  # trans_arr, src/kmer.cpp:7

Tables = Dict[Tuple[int, int, int], int]


def build(force: bool = False) -> None:
    """Compile the C oracle (and the reference, when its tree is present)."""
    if force or not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(
            os.path.join(HERE, "trew_oracle.c")):
        subprocess.check_call(["make", "-C", HERE, "_build/libtrew_oracle.so"], stdout=subprocess.DEVNULL)
    if os.path.isdir("/root/reference/src"):
        subprocess.check_call(["make", "-C", HERE, "ref"], stdout=subprocess.DEVNULL)


def seq_to_str(seq: int, k: int) -> str:
    """int_to_four, src/kmer.cpp:1886-1892."""
    return "".join(LETTERS[(seq >> (2 * (k - 1 - i))) & 3] for i in range(k))


def str_to_seq(s: str) -> int:
    v = 0
    for ch in s:
        v = (v << 2) | LETTERS.index(ch.upper())
    return v


def make_chunk(reads: Sequence[bytes]) -> Tuple[bytes, List[int]]:
    """Lay reads out like one FASTQ-free chunk: sequences separated by newlines, plus the flattened
    inclusive (st, nd) offsets a LocationVector would hold (src/kmer.h:73)."""
    locs: List[int] = []
    parts: List[bytes] = []
    pos = 0
    for r in reads:
        locs += [pos, pos + len(r) - 1]
        parts.append(r)
        parts.append(b"\n")
        pos += len(r) + 1
    return b"".join(parts), locs


class _Cfg(C.Structure):
    _fields_ = [("min_mer", C.c_int), ("max_mer", C.c_int), ("low", C.c_double), ("high", C.c_double),
                ("slice_len", C.c_int), ("emulate_pair_leak", C.c_int)]


def _export(n: int, fn, *lead) -> Tables:
    tb = (C.c_int * max(n, 1))()
    kk = (C.c_int * max(n, 1))()
    lo = (C.c_uint64 * max(n, 1))()
    hi = (C.c_uint64 * max(n, 1))()
    ct = (C.c_uint64 * max(n, 1))()
    fn(*lead, tb, kk, lo, hi, ct)
    return {(tb[i], kk[i], (hi[i] << 64) | lo[i]): ct[i] for i in range(n)}


class Oracle:
    def __init__(self, min_mer: int = 5, max_mer: int = 32, low: float = 0.5, high: float = 0.8,
                 slice_len: int = 150, emulate_pair_leak: bool = False):
        if not os.path.exists(ORACLE_SO):
            build()
        self.lib = C.CDLL(ORACLE_SO)
        self.cfg = _Cfg(min_mer, max_mer, low, high, slice_len, int(emulate_pair_leak))
        L = self.lib
        L.orc_tables_new.restype = C.c_void_p
        L.orc_tables_free.argtypes = [C.c_void_p]
        L.orc_tables_clear.argtypes = [C.c_void_p]
        L.orc_tables_size.argtypes = [C.c_void_p]
        L.orc_tables_export.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        L.orc_scan_chunk.argtypes = [C.POINTER(_Cfg), C.c_int, C.c_char_p, C.POINTER(C.c_int), C.c_int,
                                     C.c_char_p, C.POINTER(C.c_int), C.c_int, C.c_void_p]
        L.orc_k_mer_check.argtypes = [C.POINTER(_Cfg), C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.POINTER(C.c_int), C.POINTER(C.c_uint64), C.c_void_p]
        for name in ("orc_canon_c", "orc_crc_c"):
            getattr(L, name).argtypes = [C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_uint64)]
        L.orc_homo_c.argtypes = [C.c_uint64, C.c_uint64, C.c_int]
        L.orc_period_stats.argtypes = [C.POINTER(_Cfg), C.c_char_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 5

    def scan(self, mode: int, reads1: Sequence[bytes], reads2: Optional[Sequence[bytes]] = None) -> Tables:
        t = self.lib.orc_tables_new()
        try:
            b1, l1 = make_chunk(reads1)
            a1 = (C.c_int * max(len(l1), 1))(*l1)
            if mode == 1:
                b2, l2 = make_chunk(reads2 or [])
                a2 = (C.c_int * max(len(l2), 1))(*l2)
                self.lib.orc_scan_chunk(C.byref(self.cfg), 1, b1, a1, len(l1) // 2, b2, a2, len(l2) // 2, t)
            else:
                self.lib.orc_scan_chunk(C.byref(self.cfg), mode, b1, a1, len(l1) // 2, None, None, 0, t)
            return _export(self.lib.orc_tables_size(t), self.lib.orc_tables_export, t)
        finally:
            self.lib.orc_tables_free(t)

    def k_mer_check(self, seq: bytes, st: int, nd: int, kmin: int, kmax: int):
        t = self.lib.orc_tables_new()
        try:
            out = (C.c_int * 2)()
            sq = (C.c_uint64 * 4)()
            self.lib.orc_k_mer_check(C.byref(self.cfg), seq, st, nd, kmin, kmax, out, sq, t)
            em = _export(self.lib.orc_tables_size(t), self.lib.orc_tables_export, t)
            return out[0], out[1], (sq[1] << 64) | sq[0], (sq[3] << 64) | sq[2], em
        finally:
            self.lib.orc_tables_free(t)

    def period_stats(self, seq: bytes, st: int, nd: int, k: int) -> Tuple[int, int, int, int]:
        """(T, M, S, n_classes) of period k over seq[st..nd] (inclusive): valid k-windows, the largest rotation class's
        count, that class (the first to reach the maximum) and the number of classes."""
        T, M, n = C.c_int(0), C.c_int(0), C.c_int(0)
        lo, hi = C.c_uint64(0), C.c_uint64(0)
        self.lib.orc_period_stats(C.byref(self.cfg), seq, st, nd, k, C.byref(T), C.byref(M), C.byref(lo), C.byref(hi), C.byref(n))
        return T.value, M.value, (hi.value << 64) | lo.value, n.value

    @staticmethod
    def need(T: int, B: float) -> int:
        """The smallest M with (double)M / T >= B (build_thr's threshold table); T + 1 when no M reaches it."""
        M = max(0, int(B * T) - 2)
        while M <= T and M / T < B:
            M += 1
        return M

    def canon(self, seq: int, k: int) -> int:
        o = (C.c_uint64 * 2)()
        self.lib.orc_canon_c(seq & (2 ** 64 - 1), seq >> 64, k, o)
        return (o[1] << 64) | o[0]

    def crc(self, seq: int, k: int) -> int:
        o = (C.c_uint64 * 2)()
        self.lib.orc_crc_c(seq & (2 ** 64 - 1), seq >> 64, k, o)
        return (o[1] << 64) | o[0]

    def homo(self, seq: int, k: int) -> bool:
        return bool(self.lib.orc_homo_c(seq & (2 ** 64 - 1), seq >> 64, k))


def reference_available() -> bool:
    return os.path.exists(REF_SO)


class Reference:
    """The compiled reference (process-global state: one configuration at a time)."""

    def __init__(self, min_mer: int = 5, max_mer: int = 32, low: float = 0.5, high: float = 0.8,
                 slice_len: int = 150, table_max_mer: int = 8):
        self.lib = C.CDLL(REF_SO)
        L = self.lib
        L.ref_init.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int]
        L.ref_scan.argtypes = [C.c_int, C.c_char_p, C.c_long, C.POINTER(C.c_int), C.c_int,
                               C.c_char_p, C.c_long, C.POINTER(C.c_int), C.c_int]
        L.ref_result_copy.argtypes = [C.c_void_p] * 5
        L.ref_k_mer_check.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int),
                                      C.POINTER(C.c_uint64)]
        for name in ("ref_get_rot_seq", "ref_rot_reverse_complement"):
            getattr(L, name).argtypes = [C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_uint64)]
        L.ref_get_repeat_check.argtypes = [C.c_uint64, C.c_uint64, C.c_int]
        self.args = (min_mer, max_mer, table_max_mer, low, high, slice_len)
        self.activate()

    def activate(self) -> None:
        self.lib.ref_init(*self.args)

    def scan(self, mode: int, reads1: Sequence[bytes], reads2: Optional[Sequence[bytes]] = None) -> Tables:
        self.activate()
        b1, l1 = make_chunk(reads1)
        a1 = (C.c_int * max(len(l1), 1))(*l1)
        if mode == 1:
            b2, l2 = make_chunk(reads2 or [])
            a2 = (C.c_int * max(len(l2), 1))(*l2)
            n = self.lib.ref_scan(1, b1, len(b1), a1, len(l1) // 2, b2, len(b2), a2, len(l2) // 2)
        else:
            n = self.lib.ref_scan(mode, b1, len(b1), a1, len(l1) // 2, None, 0, None, 0)
        return _export(n, self.lib.ref_result_copy)

    def k_mer_check(self, seq: bytes, st: int, nd: int, kmin: int, kmax: int):
        self.activate()
        out = (C.c_int * 2)()
        sq = (C.c_uint64 * 4)()
        n = self.lib.ref_k_mer_check(seq, st, nd, kmin, kmax, out, sq)
        em = _export(n, self.lib.ref_result_copy)
        return out[0], out[1], (sq[1] << 64) | sq[0], (sq[3] << 64) | sq[2], em

    def canon(self, seq: int, k: int) -> int:
        o = (C.c_uint64 * 2)()
        self.lib.ref_get_rot_seq(seq & (2 ** 64 - 1), seq >> 64, k, o)
        return (o[1] << 64) | o[0]

    def crc(self, seq: int, k: int) -> int:
        o = (C.c_uint64 * 2)()
        self.lib.ref_rot_reverse_complement(seq & (2 ** 64 - 1), seq >> 64, k, o)
        return (o[1] << 64) | o[0]

    def homo(self, seq: int, k: int) -> bool:
        return bool(self.lib.ref_get_repeat_check(seq & (2 ** 64 - 1), seq >> 64, k))


def format_tables(t: Tables) -> List[str]:
    return ["%s %d %s %d" % (TABLE_NAMES[tb], k, seq_to_str(s, k), c) for (tb, k, s), c in sorted(t.items())]
