"""ctypes front-end of the CPU scan oracle (scan_oracle/scan_oracle.c): the scan of migrate_actions over
LSMTree::iter_filter, restated on the CPU.

TEST INFRASTRUCTURE ONLY, like the compaction oracle (oracle/): importable from tests/ and tools/; the product package
(dbeel_b200/) never imports this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libscan_oracle.so")
_SOURCES = [os.path.join(_HERE, "scan_oracle.c"), os.path.join(_HERE, "..", "oracle", "dbeel_oracle.c")]

SCAN_REFERENCE, SCAN_EXACT = 0, 1
SCAN_END, SCAN_DECODE, SCAN_READ = 0, 1, 2


class _Run(C.Structure):
    _fields_ = [("data", C.c_void_p), ("data_len", C.c_uint64), ("index", C.c_void_p), ("index_len", C.c_uint64)]


class _Out(C.Structure):
    _fields_ = [("data", C.c_void_p), ("data_cap", C.c_uint64), ("data_len", C.c_uint64),
                ("index", C.c_void_p), ("index_cap", C.c_uint64), ("index_len", C.c_uint64),
                ("bloom", C.c_void_p), ("bloom_cap", C.c_uint64), ("bloom_len", C.c_uint64),
                ("items_written", C.c_uint64)]


def build(force: bool = False) -> str:
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(_LIB_PATH) < os.path.getmtime(s) for s in _SOURCES):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libscan_oracle.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        L.orc_scan_ranges.restype = C.c_int
        L.orc_scan_ranges.argtypes = [C.POINTER(_Run), C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(_Out),
                                      C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
        L.orc_between_cmp.restype = C.c_int
        L.orc_between_cmp.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        _lib = L
    return _lib


def _u8(a) -> np.ndarray:
    if isinstance(a, np.ndarray):
        assert a.dtype == np.uint8 and a.flags.c_contiguous
        return a
    return np.frombuffer(bytes(a), dtype=np.uint8)


def between_cmp(hash_: int, start: int, end: int, mode: int = SCAN_REFERENCE) -> bool:
    return bool(lib().orc_between_cmp(hash_, start, end, mode))


def scan_ranges(tables: Sequence[Tuple[object, object]], ranges: Sequence[Tuple[int, int]], mode: int = SCAN_REFERENCE):
    """tables = [(data, index)] in iteration order, ranges = [(start, end)].  Returns (data, index, per_range, stop):
    per_range = [{data_off, data_len, index_off, index_len, items}] (the dbeel_flush_table fields), stop = (table, reason,
    record) with table -1 when the scan ran to the end."""
    keep = [(_u8(d), _u8(i)) for d, i in tables]
    arr = (_Run * max(1, len(keep)))()
    for j, (d, i) in enumerate(keep):
        arr[j] = _Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
    rng = np.ascontiguousarray(np.array(ranges, dtype=np.uint32).reshape(-1, 2))
    data_cap = sum(d.size for d, _ in keep)
    index_cap = 16 * sum(i.size // 16 for _, i in keep)
    od, oi = np.empty(max(1, data_cap), np.uint8), np.empty(max(1, index_cap), np.uint8)
    out = _Out(od.ctypes.data, data_cap, 0, oi.ctypes.data, index_cap, 0, None, 0, 0, 0)
    pr = np.zeros((max(1, len(rng)), 5), np.uint64)
    st, sr, sc = C.c_int32(), C.c_uint32(), C.c_uint64()
    rc = lib().orc_scan_ranges(arr, len(keep), rng.ctypes.data if rng.size else None, len(rng), mode, C.byref(out),
                               pr.ctypes.data, C.byref(st), C.byref(sr), C.byref(sc))
    if rc:
        raise RuntimeError(f"orc_scan_ranges rc={rc}")
    rows = [dict(data_off=int(r[0]), data_len=int(r[1]), index_off=int(r[2]), index_len=int(r[3]), items=int(r[4]))
            for r in pr[:len(rng)]]
    return od[:out.data_len], oi[:out.index_len], rows, (int(st.value), int(sr.value), int(sc.value))
