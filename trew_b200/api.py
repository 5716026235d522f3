"""ctypes binding of libtrew_b200.so -- the host-side mirror used by tests, bench.py and smoke().

The product path is the C ABI in include/trew_b200.h (C++ host code + CUDA kernels); this module only
marshals arguments.  It fails loudly when the library is missing or no CUDA device is usable: there is
no CPU fallback, and nothing here imports the oracle.

Reference interface mirrored (paths into the reference tree):
  DeviceContext.submit_chunk   <-> QueueData / PairQueueData pushed to buffer_task* (src/kmer.h:93-103)
  DeviceContext.finish         <-> the six ResultMaps summed by process_output (src/kmer.cpp:1486-1515)
  Report                       <-> process_output / final_process_output (src/kmer.cpp:1478-1634, 2571-2761)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TREW_B200_LIB", os.path.join(HERE, "libtrew_b200.so"))  # override: experiments only
CLI_PATH = os.path.join(HERE, "trew")

MODE_SHORT, MODE_PAIR, MODE_LONG = 0, 1, 2
TABLE_NAMES = ("F_h", "F_l", "B_h", "B_l", "O_h", "O_l")

Tables = Dict[Tuple[int, int, int], int]


class TrewError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__("trew_b200 status %d: %s" % (status, message))
        self.status = status


class Config(C.Structure):
    _fields_ = [("mode", C.c_int32), ("min_mer", C.c_int32), ("max_mer", C.c_int32), ("slice_length", C.c_int32),
                ("low_baseline", C.c_double), ("high_baseline", C.c_double), ("device", C.c_int32),
                ("table_log2_slots", C.c_int32), ("n_staging", C.c_int32), ("host_threads", C.c_int32),
                ("staging_bytes", C.c_uint64)]


class Batch(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("max_read_len", C.c_uint32), ("bit_off", C.POINTER(C.c_uint32)),
                ("hi", C.POINTER(C.c_uint32)), ("lo", C.POINTER(C.c_uint32)), ("val", C.POINTER(C.c_uint32))]


class Entry(C.Structure):
    _fields_ = [("seq_lo", C.c_uint64), ("seq_hi", C.c_uint64), ("count", C.c_uint64), ("table", C.c_int32),
                ("k", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("reads", C.c_uint64), ("bases", C.c_uint64), ("units", C.c_uint64), ("survivors", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("device_ms", C.c_double), ("host_pack_bytes", C.c_uint64), ("host_pack_ms", C.c_double)]


# every symbol include/trew_b200.h declares (tests/test_abi.py checks the library exports all of them)
ABI_SYMBOLS = [
    "trew_abi_version", "trew_status_string", "trew_dev_create", "trew_dev_destroy", "trew_dev_last_error",
    "trew_dev_submit_chunk", "trew_dev_submit_packed", "trew_dev_upload", "trew_dev_scan_resident",
    "trew_dev_free_resident", "trew_dev_last_resident_ms", "trew_dev_sync", "trew_dev_finish",
    "trew_dev_export_device", "trew_dev_reset", "trew_dev_get_stats", "trew_pack_bound", "trew_pack_reads",
    "trew_synth_resident", "trew_dev_timer_start", "trew_dev_timer_stop", "trew_dev_kernel_times",
    "trew_dev_process_file", "trew_ingest_file", "trew_report_create", "trew_report_destroy", "trew_report_add_file",
    "trew_report_finish", "trew_dev_export_rows", "trew_dev_merge_rows", "trew_dev_reserve", "trew_dev_finish_merged",
    "trew_pack_reads_ranges", "trew_report_text", "trew_synth_resident_ex", "trew_multi_create", "trew_multi_destroy",
    "trew_multi_device_count", "trew_multi_last_error", "trew_multi_submit_chunk", "trew_multi_process_file",
    "trew_multi_reset", "trew_multi_finish", "trew_multi_get_stats", "trew_multi_ctx", "trew_dev_set_report_filter",
    "trew_multi_set_report_filter", "trew_dev_enable_unit_records", "trew_dev_unit_records", "trew_multi_enable_unit_records",
    "trew_multi_unit_records", "trew_check_batch",
]

# trew_unit_record: one unit's adds to one (table, k, seq), sorted by (unit, table, k, seq_hi, seq_lo)
UNIT_RECORD_DTYPE = np.dtype([("unit", "<u8"), ("seq_lo", "<u8"), ("seq_hi", "<u8"), ("count", "<u4"), ("table", "u1"),
                              ("k", "u1"), ("reserved", "<u2")])
UnitRecords = Dict[Tuple[int, int, int, int], int]


def unit_records_dict(recs: np.ndarray) -> UnitRecords:
    """A unit_records() array as {(unit, table, k, seq): count}."""
    return {(int(r["unit"]), int(r["table"]), int(r["k"]), (int(r["seq_hi"]) << 64) | int(r["seq_lo"])): int(r["count"])
            for r in recs}


def _records_array(p: C.c_void_p, n: int) -> np.ndarray:
    if n == 0:
        return np.zeros(0, dtype=UNIT_RECORD_DTYPE)
    buf = (C.c_char * (n * UNIT_RECORD_DTYPE.itemsize)).from_address(p.value)
    return np.frombuffer(buf, dtype=UNIT_RECORD_DTYPE, count=n).copy()

CHUNK_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_uint32, C.c_void_p,
                        C.POINTER(C.c_int32), C.c_uint32)

_lib = None


def load_library() -> C.CDLL:
    """Load libtrew_b200.so (built in-tree by `make -C trew_b200/csrc`).  No fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TrewError(2, "%s not built: run `python -c 'import __graft_entry__ as g; g.build()'`" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.trew_status_string.restype = C.c_char_p
    L.trew_status_string.argtypes = [C.c_int]
    L.trew_dev_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    L.trew_dev_destroy.argtypes = [C.c_void_p]
    L.trew_dev_destroy.restype = None
    L.trew_dev_last_error.argtypes = [C.c_void_p]
    L.trew_dev_last_error.restype = C.c_char_p
    L.trew_dev_submit_chunk.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32]
    L.trew_dev_submit_packed.argtypes = [C.c_void_p, C.POINTER(Batch)]
    L.trew_dev_upload.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(C.c_void_p)]
    L.trew_check_batch.argtypes = [C.c_int, C.POINTER(Batch)]
    L.trew_dev_scan_resident.argtypes = [C.c_void_p, C.c_void_p]
    L.trew_dev_free_resident.argtypes = [C.c_void_p, C.c_void_p]
    L.trew_dev_free_resident.restype = None
    L.trew_dev_last_resident_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    L.trew_dev_sync.argtypes = [C.c_void_p]
    L.trew_dev_finish.argtypes = [C.c_void_p, C.POINTER(C.POINTER(Entry)), C.POINTER(C.c_uint64)]
    L.trew_dev_export_device.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.trew_dev_export_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.trew_dev_merge_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    L.trew_dev_reserve.argtypes = [C.c_void_p, C.c_uint64]
    L.trew_dev_finish_merged.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_uint32,
                                         C.POINTER(C.POINTER(Entry)), C.POINTER(C.c_uint64)]
    L.trew_dev_reset.argtypes = [C.c_void_p]
    L.trew_dev_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.trew_pack_bound.argtypes = [C.c_uint32, C.c_uint64]
    L.trew_pack_bound.restype = C.c_size_t
    L.trew_pack_reads.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.POINTER(Batch)]
    L.trew_pack_reads_ranges.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t,
                                         C.POINTER(Batch), C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.trew_dev_process_file.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_int]
    L.trew_synth_resident.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                      C.c_uint32, C.POINTER(C.c_void_p)]
    L.trew_synth_resident_ex.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                         C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
    L.trew_multi_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_void_p)]
    L.trew_multi_destroy.argtypes = [C.c_void_p]
    L.trew_multi_destroy.restype = None
    L.trew_multi_device_count.argtypes = [C.c_void_p]
    L.trew_multi_last_error.argtypes = [C.c_void_p]
    L.trew_multi_last_error.restype = C.c_char_p
    L.trew_multi_submit_chunk.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32]
    L.trew_multi_process_file.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_int]
    L.trew_multi_reset.argtypes = [C.c_void_p]
    L.trew_multi_finish.argtypes = [C.c_void_p, C.POINTER(C.POINTER(Entry)), C.POINTER(C.c_uint64)]
    L.trew_multi_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.trew_multi_ctx.argtypes = [C.c_void_p, C.c_int32]
    L.trew_multi_ctx.restype = C.c_void_p
    L.trew_dev_set_report_filter.argtypes = [C.c_void_p, C.c_uint32]
    L.trew_multi_set_report_filter.argtypes = [C.c_void_p, C.c_uint32]
    L.trew_dev_enable_unit_records.argtypes = [C.c_void_p, C.c_uint64]
    L.trew_dev_unit_records.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.trew_multi_enable_unit_records.argtypes = [C.c_void_p, C.c_uint64]
    L.trew_multi_unit_records.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.trew_dev_timer_start.argtypes = [C.c_void_p]
    L.trew_dev_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    L.trew_dev_kernel_times.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                        C.POINTER(C.c_uint64)]
    L.trew_ingest_file.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_uint64, CHUNK_SINK,
                                   C.c_void_p, C.c_char_p, C.c_size_t]
    L.trew_report_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.trew_report_destroy.argtypes = [C.c_void_p]
    L.trew_report_destroy.restype = None
    L.trew_report_add_file.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint64]
    L.trew_report_finish.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t)]
    _lib = L
    return L


def make_chunk(reads: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """Sequences laid out newline-separated plus their inclusive (st, nd) offsets -- one QueueData."""
    lens = np.fromiter((len(r) for r in reads), dtype=np.int64, count=len(reads))
    buf = np.frombuffer(b"\n".join(reads) + b"\n", dtype=np.uint8)
    st = np.zeros(len(reads), dtype=np.int64)
    if len(reads) > 1:
        st[1:] = np.cumsum(lens[:-1] + 1)
    locs = np.empty((len(reads), 2), dtype=np.int32)
    locs[:, 0] = st
    locs[:, 1] = st + lens - 1
    return buf, locs


def matrix_chunk(mat: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Fixed-length ASCII matrix (n x L, uint8) -> newline-separated chunk + offsets, vectorised."""
    n, L = mat.shape
    buf = np.empty((n, L + 1), dtype=np.uint8)
    buf[:, :L] = mat
    buf[:, L] = 10
    st = np.arange(n, dtype=np.int64) * (L + 1)
    locs = np.empty((n, 2), dtype=np.int32)
    locs[:, 0] = st
    locs[:, 1] = st + L - 1
    return buf.reshape(-1), locs


class PackedBatch:
    """A packed batch in host memory (owner of the buffer the trew_batch pointers point into)."""

    def __init__(self, buf: np.ndarray, locs: np.ndarray, n_ranges: int = 0, n_threads: int = 1, want_invalid: bool = False,
                 no_val: bool = False, buf2: Optional[np.ndarray] = None, locs2: Optional[np.ndarray] = None):
        """n_ranges > 0 packs through trew_pack_reads_ranges (concurrent ranges, optional invalid-base list in
        self.invalid, no_val = TREW_PACK_NO_VAL); otherwise through the single-threaded trew_pack_reads."""
        L = load_library()
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        locs = np.ascontiguousarray(locs, dtype=np.int32).reshape(-1, 2)
        n = locs.shape[0]
        lens = (locs[:, 1].astype(np.int64) - locs[:, 0].astype(np.int64) + 1).clip(min=0)
        self.n_reads = n
        self.bases = int(lens.sum())
        if buf2 is not None:   # a paired chunk (needs n_ranges > 0): 2 n reads, mates alternating
            buf2 = np.ascontiguousarray(buf2, dtype=np.uint8)
            locs2 = np.ascontiguousarray(locs2, dtype=np.int32).reshape(-1, 2)
            assert locs2.shape[0] == n and n_ranges > 0
            self.n_reads = 2 * n
            self.bases += int((locs2[:, 1].astype(np.int64) - locs2[:, 0].astype(np.int64) + 1).clip(min=0).sum())
        self.nbytes = L.trew_pack_bound(self.n_reads, self.bases)
        self.mem = np.zeros(self.nbytes, dtype=np.uint8)
        self.batch = Batch()
        self.invalid = None
        if n_ranges > 0:
            cap = self.bases + 64 if want_invalid else 0
            inv = np.zeros(max(cap, 1), dtype=np.uint32)
            n_inv = C.c_size_t(0)
            rc = L.trew_pack_reads_ranges(buf.ctypes.data, locs.ctypes.data, buf2.ctypes.data if buf2 is not None else None,
                                          locs2.ctypes.data if buf2 is not None else None, n, n_ranges, n_threads,
                                          1 if no_val else 0, self.mem.ctypes.data,
                                          self.nbytes, C.byref(self.batch), inv.ctypes.data if want_invalid else None, cap,
                                          C.byref(n_inv))
            if want_invalid and not rc:
                self.invalid = inv[:n_inv.value].copy()
        else:
            rc = L.trew_pack_reads(buf.ctypes.data, locs.ctypes.data, n, self.mem.ctypes.data, self.nbytes, C.byref(self.batch))
        if rc:
            raise TrewError(rc, L.trew_status_string(rc).decode())

    def planes(self) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
        """(bit_off, hi, lo, val) as numpy views -- for tests of the packer."""
        n = self.n_reads
        words = (self.bases + 31) // 32
        base = self.mem.ctypes.data

        def view(ptr, count):
            off = C.cast(ptr, C.c_void_p).value - base
            return self.mem[off:off + 4 * count].view(np.uint32)
        return (view(self.batch.bit_off, n + 1), view(self.batch.hi, words), view(self.batch.lo, words),
                view(self.batch.val, words))


class DeviceContext:
    """One GPU's scan context (trew_ctx)."""

    def __init__(self, mode: int = MODE_SHORT, min_mer: int = 5, max_mer: int = 32, low: float = 0.5, high: float = 0.8,
                 slice_length: int = 150, device: int = 0, table_log2_slots: int = 0, n_staging: int = 0,
                 host_threads: int = 0, staging_bytes: int = 0):
        self.lib = load_library()
        self.cfg = Config(mode, min_mer, max_mer, slice_length, low, high, device, table_log2_slots, n_staging,
                          host_threads, staging_bytes)
        self.ctx = C.c_void_p()
        rc = self.lib.trew_dev_create(C.byref(self.cfg), C.byref(self.ctx))
        if rc:
            self.ctx = None
            raise TrewError(rc, self.lib.trew_dev_last_error(None).decode() or self.lib.trew_status_string(rc).decode())
        self.mode = mode

    def _check(self, rc: int) -> None:
        if rc:
            raise TrewError(rc, self.lib.trew_dev_last_error(self.ctx).decode() or self.lib.trew_status_string(rc).decode())

    def close(self) -> None:
        if getattr(self, "ctx", None):
            self.lib.trew_dev_destroy(self.ctx)
            self.ctx = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def submit_chunk(self, buf1: np.ndarray, locs1: np.ndarray, buf2: Optional[np.ndarray] = None,
                     locs2: Optional[np.ndarray] = None) -> None:
        locs1 = np.ascontiguousarray(locs1, dtype=np.int32).reshape(-1, 2)
        if buf2 is not None:
            locs2 = np.ascontiguousarray(locs2, dtype=np.int32).reshape(-1, 2)
            self._check(self.lib.trew_dev_submit_chunk(self.ctx, buf1.ctypes.data, locs1.ctypes.data, locs1.shape[0],
                                                       buf2.ctypes.data, locs2.ctypes.data, locs2.shape[0]))
        else:
            self._check(self.lib.trew_dev_submit_chunk(self.ctx, buf1.ctypes.data, locs1.ctypes.data, locs1.shape[0],
                                                       None, None, 0))

    def submit_reads(self, reads1: Sequence[bytes], reads2: Optional[Sequence[bytes]] = None) -> None:
        if len(reads1) == 0:
            return
        b1, l1 = make_chunk(reads1)
        if reads2 is not None:
            b2, l2 = make_chunk(reads2)
            self.submit_chunk(b1, l1, b2, l2)
        else:
            self.submit_chunk(b1, l1)

    def submit_packed(self, pb: PackedBatch, max_read_len: Optional[int] = None) -> None:
        """max_read_len, when given, replaces the packer's value in pb.batch (at least the longest read, or TREW_ERR_ARG)."""
        if max_read_len is not None:
            pb.batch.max_read_len = max_read_len
        self._check(self.lib.trew_dev_submit_packed(self.ctx, C.byref(pb.batch)))

    def upload(self, pb: PackedBatch) -> C.c_void_p:
        h = C.c_void_p()
        self._check(self.lib.trew_dev_upload(self.ctx, C.byref(pb.batch), C.byref(h)))
        return h

    def scan_resident(self, handle) -> None:
        self._check(self.lib.trew_dev_scan_resident(self.ctx, handle))

    def last_resident_ms(self) -> float:
        ms = C.c_float()
        self._check(self.lib.trew_dev_last_resident_ms(self.ctx, C.byref(ms)))
        return ms.value

    def free_resident(self, handle) -> None:
        self.lib.trew_dev_free_resident(self.ctx, handle)

    def synth_resident(self, seed: int, n_reads: int, read_len: int = 150, tel_ppm: int = 10000, half_ppm: int = 2000,
                       n_ppm: int = 1000, sub_ppm: int = 10000, flavor: int = 0):
        """flavor 0 single reads, 1 pairs (mates of one fragment), 2 long reads with telomeric ends."""
        h = C.c_void_p()
        self._check(self.lib.trew_synth_resident_ex(self.ctx, seed, n_reads, read_len, tel_ppm, half_ppm, n_ppm, sub_ppm,
                                                    flavor, C.byref(h)))
        return h

    def timer_start(self) -> None:
        self._check(self.lib.trew_dev_timer_start(self.ctx))

    def timer_stop(self) -> float:
        ms = C.c_float()
        self._check(self.lib.trew_dev_timer_stop(self.ctx, C.byref(ms)))
        return ms.value

    def kernel_times(self) -> Tuple[float, float, float, int]:
        """(screen_ms, decide_ms, exact_ms, n_scans) accumulated over resident scans since the last call."""
        s, d, e, n = C.c_double(), C.c_double(), C.c_double(), C.c_uint64()
        self._check(self.lib.trew_dev_kernel_times(self.ctx, C.byref(s), C.byref(d), C.byref(e), C.byref(n)))
        return s.value, d.value, e.value, n.value

    def sync(self) -> None:
        self._check(self.lib.trew_dev_sync(self.ctx))

    def process_file(self, file1: str, file2: Optional[str] = None) -> None:
        gz = lambda p: int(p.endswith(".gz") or p.endswith(".bgz"))
        self._check(self.lib.trew_dev_process_file(self.ctx, file1.encode(), gz(file1),
                                                   file2.encode() if file2 else None, gz(file2) if file2 else 0))

    def finish_entries(self):
        p = C.POINTER(Entry)()
        n = C.c_uint64()
        self._check(self.lib.trew_dev_finish(self.ctx, C.byref(p), C.byref(n)))
        return p, n.value

    ENTRY_DTYPE = np.dtype([("seq_lo", "<u8"), ("seq_hi", "<u8"), ("count", "<u8"), ("table", "<i4"), ("k", "<i4")])

    def finish_view(self) -> np.ndarray:
        """The merged tables as a zero-copy structured view of the library's entry array (sorted by
        (table, k, seq)); valid until the next call that touches the tables."""
        p, n = self.finish_entries()
        if n == 0:
            return np.zeros(0, dtype=self.ENTRY_DTYPE)
        buf = (C.c_char * (n * 32)).from_address(C.addressof(p.contents))
        return np.frombuffer(buf, dtype=self.ENTRY_DTYPE, count=n)

    def finish_arrays(self) -> np.ndarray:
        """The merged tables as an (n, 4) int64 array of rows (meta = table << 8 | k, seq_lo, seq_hi, count),
        sorted by (table, k, seq).  64-bit fields are reinterpreted as signed."""
        v = self.finish_view()
        out = np.empty((v.shape[0], 4), dtype=np.uint64)
        out[:, 0] = (v["table"].astype(np.uint64) << np.uint64(8)) | v["k"].astype(np.uint64)
        out[:, 1] = v["seq_lo"]
        out[:, 2] = v["seq_hi"]
        out[:, 3] = v["count"]
        return out.view(np.int64)

    def finish(self) -> Tables:
        p, n = self.finish_entries()
        return {(p[i].table, p[i].k, (p[i].seq_hi << 64) | p[i].seq_lo): p[i].count for i in range(n)}

    def export_device(self):
        """(entries_ptr, n): device pointer to the compacted, sorted table (trew_entry rows)."""
        e, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.trew_dev_export_device(self.ctx, C.byref(e), C.byref(n)))
        return e.value, n.value

    def export_rows(self, d_rows: Optional[int] = None, capacity_rows: int = 0) -> int:
        """Compact the table; with a device pointer, also copy it there as trew_entry rows (32 bytes each).
        Returns the row count."""
        n = C.c_uint64()
        self._check(self.lib.trew_dev_export_rows(self.ctx, d_rows, capacity_rows, C.byref(n)))
        return n.value

    def merge_rows(self, d_rows: int, n_rows: int) -> None:
        """Add rows (device pointer, the format of export_rows) to this context's table."""
        self._check(self.lib.trew_dev_merge_rows(self.ctx, d_rows, n_rows))

    def finish_merged_view(self, lists) -> np.ndarray:
        """Union of this context's table and other ranks' rows (`lists` = [(device pointer, n_rows), ...]) as a
        zero-copy structured view sorted by (table, k, seq); this context's table is not modified."""
        k = len(lists)
        ptrs = (C.c_void_p * max(k, 1))(*[p for p, _ in lists])
        sizes = (C.c_uint64 * max(k, 1))(*[n for _, n in lists])
        p = C.POINTER(Entry)()
        n = C.c_uint64()
        self._check(self.lib.trew_dev_finish_merged(self.ctx, ptrs, sizes, k, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.zeros(0, dtype=self.ENTRY_DTYPE)
        buf = (C.c_char * (n.value * 32)).from_address(C.addressof(p.contents))
        return np.frombuffer(buf, dtype=self.ENTRY_DTYPE, count=n.value)

    def set_report_filter(self, min_total: int) -> None:
        """finish*() then return only the rows a one-file report can show (groups with a class total >= min_total)."""
        self._check(self.lib.trew_dev_set_report_filter(self.ctx, min_total))

    def reserve(self, expected_new_keys: int) -> None:
        """Grow the count table so that about this many more distinct keys fit at a load factor <= 1/4."""
        self._check(self.lib.trew_dev_reserve(self.ctx, expected_new_keys))

    def reset(self) -> None:
        self._check(self.lib.trew_dev_reset(self.ctx))

    def enable_unit_records(self, capacity: int) -> None:
        """Record which unit (read, or pair in paired mode) made each table add, for up to `capacity` records; 0 = off.
        Only while the table is empty (after create or reset)."""
        self._check(self.lib.trew_dev_enable_unit_records(self.ctx, capacity))

    def unit_records(self) -> np.ndarray:
        """The records so far as a structured array (UNIT_RECORD_DTYPE), sorted by (unit, table, k, seq); a copy."""
        p, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.trew_dev_unit_records(self.ctx, C.byref(p), C.byref(n)))
        return _records_array(p, n.value)

    def stats(self) -> Stats:
        s = Stats()
        self._check(self.lib.trew_dev_get_stats(self.ctx, C.byref(s)))
        return s


class MultiContext:
    """Several GPUs in one process (trew_multi): one context per device, one shared host packing pool, chunks dealt
    round-robin, exact merge on the first device at finish -- the consumer fan-out of process_kmer*
    (src/kmer.cpp:1271-1325, 1486-1515)."""

    ENTRY_DTYPE = DeviceContext.ENTRY_DTYPE

    def __init__(self, mode: int = MODE_SHORT, min_mer: int = 5, max_mer: int = 32, low: float = 0.5, high: float = 0.8,
                 slice_length: int = 150, devices: Optional[Sequence[int]] = None, table_log2_slots: int = 0,
                 n_staging: int = 0, host_threads: int = 0, staging_bytes: int = 0):
        self.lib = load_library()
        self.cfg = Config(mode, min_mer, max_mer, slice_length, low, high, 0, table_log2_slots, n_staging, host_threads,
                          staging_bytes)
        self.h = C.c_void_p()
        devs = list(devices) if devices else []
        arr = (C.c_int32 * max(1, len(devs)))(*devs)
        rc = self.lib.trew_multi_create(C.byref(self.cfg), arr if devs else None, len(devs), C.byref(self.h))
        if rc:
            self.h = None
            raise TrewError(rc, self.lib.trew_multi_last_error(None).decode() or self.lib.trew_status_string(rc).decode())
        self.mode = mode

    def _check(self, rc: int) -> None:
        if rc:
            raise TrewError(rc, self.lib.trew_multi_last_error(self.h).decode() or self.lib.trew_status_string(rc).decode())

    @property
    def device_count(self) -> int:
        return self.lib.trew_multi_device_count(self.h)

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.trew_multi_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def submit_chunk(self, buf1, locs1, buf2=None, locs2=None) -> None:
        locs1 = np.ascontiguousarray(locs1, dtype=np.int32).reshape(-1, 2)
        if buf2 is not None:
            locs2 = np.ascontiguousarray(locs2, dtype=np.int32).reshape(-1, 2)
            self._check(self.lib.trew_multi_submit_chunk(self.h, buf1.ctypes.data, locs1.ctypes.data, locs1.shape[0],
                                                         buf2.ctypes.data, locs2.ctypes.data, locs2.shape[0]))
        else:
            self._check(self.lib.trew_multi_submit_chunk(self.h, buf1.ctypes.data, locs1.ctypes.data, locs1.shape[0], None, None, 0))

    def submit_reads(self, reads1, reads2=None, chunk_reads: int = 0) -> None:
        """chunk_reads > 0 cuts the reads into chunks of that many (each chunk goes to the next device)."""
        step = chunk_reads if chunk_reads > 0 else max(1, len(reads1))
        for i in range(0, len(reads1), step):
            b1, l1 = make_chunk(reads1[i:i + step])
            if reads2 is not None:
                b2, l2 = make_chunk(reads2[i:i + step])
                self.submit_chunk(b1, l1, b2, l2)
            else:
                self.submit_chunk(b1, l1)

    def process_file(self, file1: str, file2: Optional[str] = None) -> None:
        gz = lambda p: int(p.endswith(".gz") or p.endswith(".bgz"))
        self._check(self.lib.trew_multi_process_file(self.h, file1.encode(), gz(file1), file2.encode() if file2 else None,
                                                     gz(file2) if file2 else 0))

    def set_report_filter(self, min_total: int) -> None:
        self._check(self.lib.trew_multi_set_report_filter(self.h, min_total))

    def reset(self) -> None:
        self._check(self.lib.trew_multi_reset(self.h))

    def enable_unit_records(self, capacity: int) -> None:
        """DeviceContext.enable_unit_records for every device of the group (capacity per device)."""
        self._check(self.lib.trew_multi_enable_unit_records(self.h, capacity))

    def unit_records(self) -> np.ndarray:
        """The group's records (ordinals in its submission order), united on the first device; a copy."""
        p, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.trew_multi_unit_records(self.h, C.byref(p), C.byref(n)))
        return _records_array(p, n.value)

    def finish_view(self) -> np.ndarray:
        p = C.POINTER(Entry)()
        n = C.c_uint64()
        self._check(self.lib.trew_multi_finish(self.h, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.zeros(0, dtype=self.ENTRY_DTYPE)
        buf = (C.c_char * (n.value * 32)).from_address(C.addressof(p.contents))
        return np.frombuffer(buf, dtype=self.ENTRY_DTYPE, count=n.value)

    def finish(self) -> Tables:
        v = self.finish_view()
        return {(int(r["table"]), int(r["k"]), (int(r["seq_hi"]) << 64) | int(r["seq_lo"])): int(r["count"]) for r in v}

    def stats(self) -> Stats:
        s = Stats()
        self._check(self.lib.trew_multi_get_stats(self.h, C.byref(s)))
        return s


class Report:
    """process_output + final_process_output on the host (trew_report_*)."""

    def __init__(self, min_mer: int):
        self.lib = load_library()
        self.h = C.c_void_p()
        rc = self.lib.trew_report_create(min_mer, C.byref(self.h))
        if rc:
            raise TrewError(rc, "trew_report_create")

    def add_file(self, name: str, tables: Tables) -> None:
        n = len(tables)
        arr = (Entry * max(n, 1))()
        for i, ((tb, k, seq), cnt) in enumerate(sorted(tables.items())):
            arr[i] = Entry(seq & (2 ** 64 - 1), seq >> 64, cnt, tb, k)
        rc = self.lib.trew_report_add_file(self.h, name.encode(), arr, n)
        if rc:
            raise TrewError(rc, "trew_report_add_file")

    def add_file_entries(self, name: str, entries, n: int) -> None:
        rc = self.lib.trew_report_add_file(self.h, name.encode(), entries, n)
        if rc:
            raise TrewError(rc, "trew_report_add_file")

    def finish(self) -> str:
        t = C.c_char_p()
        n = C.c_size_t()
        self.lib.trew_report_finish(self.h, C.byref(t), C.byref(n))
        return t.value.decode()

    def __del__(self):
        try:
            if self.h:
                self.lib.trew_report_destroy(self.h)
                self.h = None
        except Exception:
            pass


def ingest_records(mode: int, file1: str, file2: Optional[str] = None, slice_length: int = 150,
                   chunk_bytes: int = 0) -> Tuple[int, str, List[bytes], List[bytes]]:
    """Run the library's FASTQ reader alone; returns (status, message, sequences of file 1, of file 2)."""
    L = load_library()
    out1: List[bytes] = []
    out2: List[bytes] = []

    def sink(user, b1, l1, n1, b2, l2, n2):
        for i in range(n1):
            out1.append(C.string_at(b1 + l1[2 * i], l1[2 * i + 1] - l1[2 * i] + 1))
        for i in range(n2):
            out2.append(C.string_at(b2 + l2[2 * i], l2[2 * i + 1] - l2[2 * i] + 1))
        return 0

    gz = lambda p: int(p.endswith(".gz") or p.endswith(".bgz"))
    msg = C.create_string_buffer(512)
    cb = CHUNK_SINK(sink)
    rc = L.trew_ingest_file(mode, slice_length, file1.encode(), gz(file1), file2.encode() if file2 else None,
                            gz(file2) if file2 else 0, chunk_bytes, cb, None, msg, 512)
    return rc, msg.value.decode(), out1, out2
