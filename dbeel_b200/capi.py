"""ctypes binding of include/dbeel_compact.h -- the same C ABI a Rust `extern "C"` block
would bind (INTEGRATION.md).  There is no CPU fallback: if libdbeel_compact.so is missing or
no sm_100 device is present, this module raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DBEEL_LIB") or os.path.join(_HERE, "libdbeel_compact.so")  # DBEEL_LIB: A/B builds only

DBEEL_OK = 0
ERR_NAMES = {1: "INVALID_ARG", 2: "CAPACITY", 3: "ITEM_TOO_LARGE", 4: "CUDA", 5: "NOMEM", 6: "TOO_MANY_RUNS",
             7: "TOO_MANY_ENTRIES", 8: "UNSORTED_RUN", 9: "NO_DEVICE", 10: "BUSY", 11: "BAD_BLOOM", 12: "TREE_FULL"}
ERR_BAD_BLOOM = 11
ERR_TREE_FULL = 12
ERR_ITEM_TOO_LARGE = 3
DEFAULT_TREE_CAPACITY = 8192  # mod.rs:18
LOOKUP_REFERENCE = 0  # the reference's binary_search loop, step for step (lsm_tree.rs:605-670)
LOOKUP_EXACT = 1      # lower-bound search: every present key is found
LOOKUP_CORRUPT = 0x80000000
ERR_UNSORTED_RUN = 8
ERR_CAPACITY = 2
ERR_INVALID_ARG = 1
ERR_NO_DEVICE = 9
FLAG_VERIFY_SORTED = 0x1
FLAG_REFERENCE_READER = 0x2  # decode runs like read_next_entry (lsm_tree.rs:1158-1170): offset / key_size ignored, timestamps range-checked
DEFAULT_BLOOM_MIN_SIZE = 1_048_576
DEFAULT_BLOOM_FP = 0.01
SCAN_REFERENCE = 0  # between_cmp read literally (migration.rs:54-60): a wrapped range holds for every hash
SCAN_EXACT = 1      # a wrapped range (end < start) is [start, 2^32) u [0, end)
MAX_SCAN_RANGES = 256
SCAN_END, SCAN_DECODE, SCAN_READ = 0, 1, 2  # dbeel_scan_stop.reason

EXPORTS = ["dbeel_abi_version", "dbeel_engine_create", "dbeel_engine_destroy", "dbeel_compact_bound",
           "dbeel_compact", "dbeel_compact_stream", "dbeel_compact_device", "dbeel_compact_submit", "dbeel_poll", "dbeel_wait",
           "dbeel_flush", "dbeel_flush_device", "dbeel_flush_many", "dbeel_flush_many_device",
           "dbeel_get_many", "dbeel_get_many_device", "dbeel_wal_flush", "dbeel_wal_flush_device",
           "dbeel_compact_many_bound", "dbeel_compact_many", "dbeel_compact_many_device",
           "dbeel_bloom_bitmap_bytes", "dbeel_bloom_k_num", "dbeel_bloom_file_size", "dbeel_host_alloc",
           "dbeel_host_free", "dbeel_last_stats", "dbeel_last_error", "dbeel_strerror",
           "dbeel_murmur3_32", "dbeel_ring_owner", "dbeel_shard_ring", "dbeel_route_device", "dbeel_flush_many_sparse_device",
           "dbeel_gpu_numa_node", "dbeel_bind_to_gpu", "dbeel_memtable_cuts_device", "dbeel_engine_stream",
           "dbeel_scan_ranges", "dbeel_scan_ranges_device", "dbeel_scan_ranges_stream"]


class Run(C.Structure):
    _fields_ = [("data", C.c_void_p), ("data_len", C.c_uint64), ("index", C.c_void_p), ("index_len", C.c_uint64)]


STREAM_READ_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p)
STREAM_WRITE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64)


class StreamIO(C.Structure):
    _fields_ = [("read", STREAM_READ_FN), ("write", STREAM_WRITE_FN), ("ctx", C.c_void_p)]


SCAN_READ_FN = STREAM_READ_FN  # (ctx, table, kind, offset, len, dst)
SCAN_WRITE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64)  # (ctx, range, kind, ...)


class ScanIO(C.Structure):
    _fields_ = [("read", SCAN_READ_FN), ("write", SCAN_WRITE_FN), ("ctx", C.c_void_p)]


class Out(C.Structure):
    _fields_ = [("data", C.c_void_p), ("data_cap", C.c_uint64), ("data_len", C.c_uint64),
                ("index", C.c_void_p), ("index_cap", C.c_uint64), ("index_len", C.c_uint64),
                ("bloom", C.c_void_p), ("bloom_cap", C.c_uint64), ("bloom_len", C.c_uint64),
                ("items_written", C.c_uint64)]


class FlushTable(C.Structure):
    _fields_ = [("data_off", C.c_uint64), ("data_len", C.c_uint64), ("index_off", C.c_uint64),
                ("index_len", C.c_uint64), ("items", C.c_uint64)]


class Job(C.Structure):
    _fields_ = [("runs", C.POINTER(Run)), ("n_runs", C.c_uint32), ("keep_tombstones", C.c_int32), ("bloom_seed", C.c_char_p)]


class JobResult(C.Structure):
    _fields_ = [("data_off", C.c_uint64), ("data_len", C.c_uint64), ("index_off", C.c_uint64), ("index_len", C.c_uint64),
                ("bloom_off", C.c_uint64), ("bloom_len", C.c_uint64), ("items_written", C.c_uint64)]


class Table(C.Structure):
    _fields_ = [("data", C.c_void_p), ("data_len", C.c_uint64), ("index", C.c_void_p), ("index_len", C.c_uint64),
                ("bloom", C.c_void_p), ("bloom_len", C.c_uint64)]


class HashRange(C.Structure):
    _fields_ = [("start", C.c_uint32), ("end", C.c_uint32)]


class ScanStop(C.Structure):
    _fields_ = [("table", C.c_int32), ("reason", C.c_uint32), ("record", C.c_uint64)]


class LookupResult(C.Structure):
    _fields_ = [("table", C.c_int32), ("bloom_rejects", C.c_uint32), ("record", C.c_uint64)]


LOOKUP_DTYPE = np.dtype([("table", "<i4"), ("bloom_rejects", "<u4"), ("record", "<u8")])


def pack_keys(keys: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """Query keys in the layout dbeel_get_many takes: (bytes back to back, n + 1 offsets)."""
    off = np.zeros(len(keys) + 1, dtype=np.uint64)
    if keys:
        off[1:] = np.cumsum(np.fromiter((len(k) for k in keys), dtype=np.uint64, count=len(keys)))
    blob = np.frombuffer(b"".join(keys), dtype=np.uint8) if keys else np.zeros(0, np.uint8)
    return blob, off


class Opts(C.Structure):
    _fields_ = [("keep_tombstones", C.c_int32), ("flags", C.c_uint32), ("bloom_min_size", C.c_uint64),
                ("bloom_fp", C.c_double), ("bloom_seed", C.c_char_p)]


class Stats(C.Structure):
    _fields_ = [("input_bytes", C.c_uint64), ("output_bytes", C.c_uint64), ("entries_in", C.c_uint64),
                ("entries_valid", C.c_uint64), ("entries_out", C.c_uint64), ("runs_truncated", C.c_uint32),
                ("key_prefix_len", C.c_uint32), ("merge_passes", C.c_uint32), ("kernel_launches", C.c_uint32),
                ("ms_total", C.c_float), ("ms_extract", C.c_float), ("ms_merge", C.c_float),
                ("ms_resolve", C.c_float), ("ms_gather", C.c_float), ("ms_h2d", C.c_float), ("ms_d2h", C.c_float),
                ("gather_bytes", C.c_uint64), ("partitions", C.c_uint32), ("index_repaired", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class DbeelError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"dbeel error {code} ({ERR_NAMES.get(code, '?')}): {msg}")
        self.code = code


_lib = None


def lib():
    """The loaded library.  Fails loudly when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH) and "DBEEL_LIB" not in os.environ:
            try:  # a fresh checkout: the .so is git-ignored; build it in-tree if the toolkit is here
                from . import _build
                _build.build()
            except Exception as ex:
                raise RuntimeError(f"{LIB_PATH} is missing and could not be built ({ex}): run "
                                   "`python -m dbeel_b200._build` where nvcc is. There is no CPU fallback "
                                   "for the compaction path.") from ex
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing. There is no CPU fallback for the compaction path.")
        L = C.CDLL(LIB_PATH)
        L.dbeel_abi_version.restype = C.c_int
        L.dbeel_engine_create.restype = C.c_int
        L.dbeel_engine_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.dbeel_engine_stream.restype = C.c_void_p
        L.dbeel_engine_stream.argtypes = [C.c_void_p]
        L.dbeel_engine_destroy.restype = None
        L.dbeel_engine_destroy.argtypes = [C.c_void_p]
        L.dbeel_compact_bound.restype = C.c_int
        L.dbeel_compact_bound.argtypes = [C.POINTER(Run), C.c_uint32, C.POINTER(Opts)] + [C.POINTER(C.c_uint64)] * 3
        for name in ("dbeel_compact", "dbeel_compact_device"):
            f = getattr(L, name)
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.POINTER(Run), C.c_uint32, C.POINTER(Opts), C.POINTER(Out)]
        L.dbeel_compact_stream.restype = C.c_int
        L.dbeel_compact_stream.argtypes = [C.c_void_p, C.POINTER(Run), C.c_uint32, C.POINTER(Opts), C.POINTER(StreamIO), C.POINTER(Out)]
        L.dbeel_compact_submit.restype = C.c_int
        L.dbeel_compact_submit.argtypes = [C.c_void_p, C.POINTER(Run), C.c_uint32, C.POINTER(Opts), C.POINTER(Out)]
        L.dbeel_poll.restype = C.c_int
        L.dbeel_poll.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        L.dbeel_wait.restype = C.c_int
        L.dbeel_wait.argtypes = [C.c_void_p]
        for name in ("dbeel_flush", "dbeel_flush_device"):
            f = getattr(L, name)
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.POINTER(Run), C.POINTER(Out)]
        for name in ("dbeel_flush_many", "dbeel_flush_many_device"):
            f = getattr(L, name)
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.POINTER(Run), C.c_uint32, C.POINTER(Out), C.POINTER(FlushTable)]
        for name in ("dbeel_get_many", "dbeel_get_many_device"):
            f = getattr(L, name)
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.POINTER(Table), C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                          C.c_void_p]
        L.dbeel_compact_many_bound.restype = C.c_int
        L.dbeel_compact_many_bound.argtypes = [C.POINTER(Job), C.c_uint32, C.c_uint64, C.c_double] + [C.POINTER(C.c_uint64)] * 3
        for name in ("dbeel_compact_many", "dbeel_compact_many_device"):
            f = getattr(L, name)
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.POINTER(Job), C.c_uint32, C.c_uint64, C.c_double, C.POINTER(Out), C.POINTER(JobResult)]
        for name in ("dbeel_wal_flush", "dbeel_wal_flush_device"):
            f = getattr(L, name)
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(Out)]
        L.dbeel_bloom_bitmap_bytes.restype = C.c_uint64
        L.dbeel_bloom_bitmap_bytes.argtypes = [C.c_uint64, C.c_double]
        L.dbeel_bloom_k_num.restype = C.c_uint32
        L.dbeel_bloom_k_num.argtypes = [C.c_uint64, C.c_uint64]
        L.dbeel_bloom_file_size.restype = C.c_uint64
        L.dbeel_bloom_file_size.argtypes = [C.c_uint64, C.c_double]
        L.dbeel_host_alloc.restype = C.c_void_p
        L.dbeel_host_alloc.argtypes = [C.c_uint64]
        L.dbeel_host_free.restype = None
        L.dbeel_host_free.argtypes = [C.c_void_p]
        L.dbeel_last_stats.restype = C.c_int
        L.dbeel_last_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.dbeel_last_error.restype = C.c_char_p
        L.dbeel_last_error.argtypes = [C.c_void_p]
        L.dbeel_strerror.restype = C.c_char_p
        L.dbeel_strerror.argtypes = [C.c_int]
        L.dbeel_gpu_numa_node.restype = C.c_int
        L.dbeel_gpu_numa_node.argtypes = [C.c_int]
        L.dbeel_bind_to_gpu.restype = C.c_int
        L.dbeel_bind_to_gpu.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.dbeel_murmur3_32.restype = C.c_uint32
        L.dbeel_murmur3_32.argtypes = [C.c_char_p, C.c_uint64, C.c_uint32]
        L.dbeel_ring_owner.restype = C.c_uint32
        L.dbeel_ring_owner.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        L.dbeel_shard_ring.restype = C.c_int
        L.dbeel_shard_ring.argtypes = [C.c_char_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.dbeel_route_device.restype = C.c_int
        L.dbeel_route_device.argtypes = [C.c_void_p, C.POINTER(Run), C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
        L.dbeel_memtable_cuts_device.restype = C.c_int
        L.dbeel_memtable_cuts_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                 C.c_uint32]
        L.dbeel_flush_many_sparse_device.restype = C.c_int
        L.dbeel_flush_many_sparse_device.argtypes = [C.c_void_p, C.POINTER(Run), C.c_uint32, C.c_uint64, C.POINTER(Out),
                                                     C.POINTER(FlushTable)]
        for name in ("dbeel_scan_ranges", "dbeel_scan_ranges_device"):
            f = getattr(L, name)
            f.restype = C.c_int
            f.argtypes = [C.c_void_p, C.POINTER(Run), C.c_uint32, C.POINTER(HashRange), C.c_uint32, C.c_uint32, C.POINTER(Out),
                          C.POINTER(FlushTable), C.POINTER(ScanStop)]
        L.dbeel_scan_ranges_stream.restype = C.c_int
        L.dbeel_scan_ranges_stream.argtypes = [C.c_void_p, C.POINTER(Run), C.c_uint32, C.POINTER(HashRange), C.c_uint32, C.c_uint32,
                                               C.POINTER(ScanIO), C.c_uint64, C.POINTER(FlushTable), C.POINTER(ScanStop)]
        _lib = L
    return _lib


def _u8(a) -> np.ndarray:
    if isinstance(a, np.ndarray):
        if a.dtype != np.uint8 or not a.flags.c_contiguous:
            a = np.ascontiguousarray(a, dtype=np.uint8)
        return a
    return np.frombuffer(bytes(a), dtype=np.uint8)


def make_opts(keep_tombstones: bool = False, bloom_min_size: int = DEFAULT_BLOOM_MIN_SIZE,
              bloom_fp: float = DEFAULT_BLOOM_FP, seed: Optional[bytes] = None, flags: int = 0) -> Opts:
    if seed is not None and len(seed) != 32:
        raise ValueError("bloom seed must be 32 bytes")
    return Opts(int(keep_tombstones), flags, bloom_min_size, bloom_fp, seed)


def compact_bound(runs: Sequence[Tuple[int, int]], opts: Opts) -> Tuple[int, int, int]:
    """runs: (data_len, index_len) pairs -> (data_cap, index_cap, bloom_cap)."""
    arr = (Run * max(1, len(runs)))()
    for j, (dl, il) in enumerate(runs):
        arr[j] = Run(None, dl, None, il)
    d, i, b = C.c_uint64(), C.c_uint64(), C.c_uint64()
    rc = lib().dbeel_compact_bound(arr, len(runs), C.byref(opts), C.byref(d), C.byref(i), C.byref(b))
    if rc:
        raise DbeelError(rc, "dbeel_compact_bound")
    return d.value, i.value, b.value


class PinnedBuffer:
    """dbeel_host_alloc'ed memory exposed as a numpy uint8 array."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        self.ptr = lib().dbeel_host_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError(f"dbeel_host_alloc({nbytes})")
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_uint8)), shape=(max(1, self.nbytes),))[:self.nbytes]

    def free(self):
        if self.ptr:
            self.array = None
            lib().dbeel_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """One compaction engine bound to one GPU (dbeel_engine_create)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        rc = lib().dbeel_engine_create(device, C.byref(self._h))
        if rc:
            raise DbeelError(rc, f"dbeel_engine_create({device}): {lib().dbeel_strerror(rc).decode()}")
        self.device = device

    def close(self):
        if self._h:
            lib().dbeel_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc:
            raise DbeelError(rc, f"{what}: {lib().dbeel_last_error(self._h).decode()}")

    def stream_ptr(self) -> int:
        """The engine's cudaStream_t as an integer (torch.cuda.ExternalStream(ptr) wraps it)."""
        return int(lib().dbeel_engine_stream(self._h) or 0)

    def stats(self) -> dict:
        s = Stats()
        lib().dbeel_last_stats(self._h, C.byref(s))
        return s.as_dict()

    # ---- host buffers (numpy) -------------------------------------------------------
    def compact(self, runs: Sequence[Tuple[object, object]], keep_tombstones: bool = False,
                bloom_min_size: int = DEFAULT_BLOOM_MIN_SIZE, seed: Optional[bytes] = None,
                bloom_fp: float = DEFAULT_BLOOM_FP, flags: int = 0, out_buffers=None):
        """dbeel_compact: returns (data, index, bloom|None, items_written) as numpy uint8 arrays."""
        keep = [(_u8(d), _u8(i)) for d, i in runs]
        arr = (Run * max(1, len(keep)))()
        for j, (d, i) in enumerate(keep):
            arr[j] = Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
        opts = make_opts(keep_tombstones, bloom_min_size, bloom_fp, seed, flags)
        dc, ic, bc = compact_bound([(d.size, i.size) for d, i in keep], opts)
        if out_buffers is None:
            od, oi, ob = (np.empty(max(1, dc), np.uint8), np.empty(max(1, ic), np.uint8), np.empty(max(1, bc), np.uint8))
        else:
            od, oi, ob = out_buffers
        out = Out(od.ctypes.data, dc, 0, oi.ctypes.data, ic, 0, ob.ctypes.data if bc else None, bc, 0, 0)
        self._check(lib().dbeel_compact(self._h, arr, len(keep), C.byref(opts), C.byref(out)), "dbeel_compact")
        bloom = ob[:out.bloom_len] if out.bloom_len else None
        return od[:out.data_len], oi[:out.index_len], bloom, int(out.items_written)

    def compact_stream(self, runs: Sequence[Tuple[object, object]], keep_tombstones: bool = False,
                       bloom_min_size: int = DEFAULT_BLOOM_MIN_SIZE, seed: Optional[bytes] = None, flags: int = 0,
                       fail_read_at: int = -1, fail_write_at: int = -1):
        """dbeel_compact_stream with in-memory "files": the engine pulls the runs through a read callback and pushes the
        output through a write callback (both called from several engine threads).  Returns (data, index, bloom|None,
        items_written) like compact(); fail_*_at = n makes the n-th callback call return error code 4242 (tests)."""
        keep = [(_u8(d), _u8(i)) for d, i in runs]
        arr = (Run * max(1, len(keep)))()
        for j, (d, i) in enumerate(keep):
            arr[j] = Run(None, d.size, None, i.size)
        opts = make_opts(keep_tombstones, bloom_min_size, DEFAULT_BLOOM_FP, seed, flags)
        dc, ic, bc = compact_bound([(d.size, i.size) for d, i in keep], opts)
        outs = {1: np.zeros(max(1, dc), np.uint8), 2: np.zeros(max(1, ic), np.uint8), 3: np.zeros(max(1, bc), np.uint8)}
        calls = {"r": 0, "w": 0}
        import threading
        mu = threading.Lock()

        def rd(_ctx, run, kind, off, n, dst):
            with mu:
                k = calls["r"]
                calls["r"] += 1
            if k == fail_read_at:
                return 4242
            src = keep[run][0] if kind == 1 else keep[run][1]
            if off + n > src.size:
                return 4243
            C.memmove(dst, src.ctypes.data + off, n)
            return 0

        def wr(_ctx, kind, off, src, n):
            with mu:
                k = calls["w"]
                calls["w"] += 1
            if k == fail_write_at:
                return 4242
            dst = outs.get(kind)
            if dst is None or off + n > dst.size:
                return 4244
            C.memmove(dst.ctypes.data + off, src, n)
            return 0

        io = StreamIO(STREAM_READ_FN(rd), STREAM_WRITE_FN(wr), None)
        out = Out(None, 0, 0, None, 0, 0, None, 0, 0, 0)
        self._check(lib().dbeel_compact_stream(self._h, arr, len(keep), C.byref(opts), C.byref(io), C.byref(out)), "dbeel_compact_stream")
        bloom = outs[3][:out.bloom_len] if out.bloom_len else None
        return outs[1][:out.data_len], outs[2][:out.index_len], bloom, int(out.items_written)

    def compact_async(self, runs: Sequence[Tuple[object, object]], keep_tombstones: bool = False,
                      bloom_min_size: int = DEFAULT_BLOOM_MIN_SIZE, seed: Optional[bytes] = None):
        """dbeel_compact_submit: returns a callable `reap(block)` -> None while running, else the result tuple."""
        keep = [(_u8(d), _u8(i)) for d, i in runs]
        arr = (Run * max(1, len(keep)))()
        for j, (d, i) in enumerate(keep):
            arr[j] = Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
        opts = make_opts(keep_tombstones, bloom_min_size, DEFAULT_BLOOM_FP, seed, 0)
        dc, ic, bc = compact_bound([(d.size, i.size) for d, i in keep], opts)
        od, oi, ob = np.empty(max(1, dc), np.uint8), np.empty(max(1, ic), np.uint8), np.empty(max(1, bc), np.uint8)
        out = Out(od.ctypes.data, dc, 0, oi.ctypes.data, ic, 0, ob.ctypes.data if bc else None, bc, 0, 0)
        self._check(lib().dbeel_compact_submit(self._h, arr, len(keep), C.byref(opts), C.byref(out)), "dbeel_compact_submit")
        alive = (keep, arr, opts, out, od, oi, ob)  # everything the job points at stays referenced by the closure

        def reap(block: bool = False):
            if block:
                rc = lib().dbeel_wait(self._h)
            else:
                st = C.c_int(0)
                if not lib().dbeel_poll(self._h, C.byref(st)):
                    return None
                rc = st.value
            self._check(rc, "dbeel_compact (async)")
            o = alive[3]
            bloom = ob[:o.bloom_len] if o.bloom_len else None
            return od[:o.data_len], oi[:o.index_len], bloom, int(o.items_written)

        return reap

    def flush(self, batch: Tuple[object, object]):
        """dbeel_flush: returns (data, index, items_written)."""
        d, i = _u8(batch[0]), _u8(batch[1])
        run = Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
        od, oi = np.empty(max(1, d.size), np.uint8), np.empty(max(1, i.size), np.uint8)
        out = Out(od.ctypes.data, d.size, 0, oi.ctypes.data, i.size // 16 * 16, 0, None, 0, 0, 0)
        self._check(lib().dbeel_flush(self._h, C.byref(run), C.byref(out)), "dbeel_flush")
        return od[:out.data_len], oi[:out.index_len], int(out.items_written)

    def flush_many(self, batches: Sequence[Tuple[object, object]]):
        """dbeel_flush_many: one launch sequence for all memtables; returns [(data, index, items)] per batch."""
        keep = [(_u8(d), _u8(i)) for d, i in batches]
        n = len(keep)
        arr = (Run * max(1, n))()
        for j, (d, i) in enumerate(keep):
            arr[j] = Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
        dc = sum(d.size for d, _ in keep)
        ic = sum(i.size // 16 * 16 for _, i in keep)
        od, oi = np.empty(max(1, dc), np.uint8), np.empty(max(1, ic), np.uint8)
        out = Out(od.ctypes.data, dc, 0, oi.ctypes.data, ic, 0, None, 0, 0, 0)
        table = (FlushTable * max(1, n))()
        self._check(lib().dbeel_flush_many(self._h, arr, n, C.byref(out), table), "dbeel_flush_many")
        return [(od[t.data_off:t.data_off + t.data_len], oi[t.index_off:t.index_off + t.index_len], int(t.items))
                for t in table[:n]]

    def flush_many_device(self, batches: Sequence[Tuple[int, int, int, int]], out_ptrs: Tuple[int, int, int, int]):
        """batches: (data_ptr, data_len, index_ptr, index_len) device pointers; out_ptrs: (data_ptr, data_cap,
        index_ptr, index_cap).  Returns (data_len, index_len, items, table rows as dicts)."""
        n = len(batches)
        arr = (Run * max(1, n))()
        for j, b in enumerate(batches):
            arr[j] = Run(*b)
        dp, dc, ip, ic = out_ptrs
        out = Out(dp, dc, 0, ip, ic, 0, None, 0, 0, 0)
        table = (FlushTable * max(1, n))()
        self._check(lib().dbeel_flush_many_device(self._h, arr, n, C.byref(out), table), "dbeel_flush_many_device")
        rows = [{k: int(getattr(t, k)) for k, _ in FlushTable._fields_} for t in table[:n]]
        return int(out.data_len), int(out.index_len), int(out.items_written), rows

    def flush_many_sparse_device(self, batches: Sequence[Tuple[int, int, int, int]], payload_bound: int,
                                 out_ptrs: Tuple[int, int, int, int]):
        """dbeel_flush_many_sparse_device: like flush_many_device, for slices of a routed stream (shared .data)."""
        n = len(batches)
        arr = (Run * max(1, n))()
        for j, b in enumerate(batches):
            arr[j] = Run(*b)
        dp, dc, ip, ic = out_ptrs
        out = Out(dp, dc, 0, ip, ic, 0, None, 0, 0, 0)
        table = (FlushTable * max(1, n))()
        self._check(lib().dbeel_flush_many_sparse_device(self._h, arr, n, payload_bound, C.byref(out), table),
                    "dbeel_flush_many_sparse_device")
        rows = [{k: int(getattr(t, k)) for k, _ in FlushTable._fields_} for t in table[:n]]
        return int(out.data_len), int(out.index_len), int(out.items_written), rows

    def memtable_cuts_device(self, key_hash64_ptr: int, stream_starts, capacity: int = DEFAULT_TREE_CAPACITY):
        """dbeel_memtable_cuts_device: per stream the list of cumulative arrival counts at which a full memtable ends."""
        starts = np.ascontiguousarray(stream_starts, np.uint64)
        n = starts.size - 1
        cap = int((starts[-1] - starts[0]) // max(1, capacity)) + n + 1
        cuts = np.zeros(cap, np.uint32)
        cs = np.zeros(n + 1, np.uint32)
        self._check(lib().dbeel_memtable_cuts_device(self._h, key_hash64_ptr or None, starts.ctypes.data, n, capacity, cuts.ctypes.data,
                                                     cs.ctypes.data, cap), "dbeel_memtable_cuts_device")
        return [cuts[cs[s]:cs[s + 1]].astype(np.int64) for s in range(n)]

    def route_device(self, batch: Tuple[int, int, int, int], ring: np.ndarray, out_index_ptr: int, out_index_cap: int,
                     shard_of_ptr: int = 0, out_hash64_ptr: int = 0):
        """dbeel_route_device: batch = (data_ptr, data_len, index_ptr, index_len) device pointers.  Returns (counts,
        payload bytes) per ring position as numpy u64 arrays."""
        ring = np.ascontiguousarray(ring, np.uint32)
        run = Run(*batch)
        counts = np.zeros(ring.size, np.uint64)
        nbytes = np.zeros(ring.size, np.uint64)
        self._check(lib().dbeel_route_device(self._h, C.byref(run), ring.ctypes.data, ring.size, out_index_ptr, out_index_cap,
                                             shard_of_ptr or None, out_hash64_ptr or None, counts.ctypes.data, nbytes.ctypes.data),
                    "dbeel_route_device")
        return counts, nbytes

    # ---- N1: many compactions per launch sequence -------------------------------------------
    @staticmethod
    def _jobs_array(jobs_ptrs, seeds):
        """jobs_ptrs: per job (list of (data_ptr, data_len, index_ptr, index_len), keep_tombstones)."""
        n = len(jobs_ptrs)
        arr = (Job * max(1, n))()
        keep = []
        for j, (runs, keep_t) in enumerate(jobs_ptrs):
            ra = (Run * max(1, len(runs)))()
            for k, r in enumerate(runs):
                ra[k] = Run(*r)
            keep.append(ra)
            arr[j] = Job(ra, len(runs), int(keep_t), seeds[j] if seeds is not None else None)
        return arr, keep

    def compact_many(self, jobs: Sequence[Tuple[Sequence[Tuple[object, object]], bool]],
                     bloom_min_size: int = DEFAULT_BLOOM_MIN_SIZE, seeds: Optional[Sequence[Optional[bytes]]] = None,
                     fp: float = DEFAULT_BLOOM_FP):
        """dbeel_compact_many over host buffers.  jobs: (runs, keep_tombstones) per compaction.  Returns one
        (data, index, bloom | None, items_written) per job, each what dbeel_compact would return for it."""
        hold = [[(_u8(d), _u8(i)) for d, i in runs] for runs, _ in jobs]
        ptrs = [([(d.ctypes.data, d.size, i.ctypes.data, i.size) for d, i in h], k) for h, (_, k) in zip(hold, jobs)]
        arr, keep = self._jobs_array(ptrs, seeds)
        n = len(jobs)
        dc, ic, bc = C.c_uint64(), C.c_uint64(), C.c_uint64()
        rc = lib().dbeel_compact_many_bound(arr, n, bloom_min_size, fp, C.byref(dc), C.byref(ic), C.byref(bc))
        if rc:
            raise DbeelError(rc, "dbeel_compact_many_bound")
        od, oi, ob = (np.empty(max(1, c.value), np.uint8) for c in (dc, ic, bc))
        out = Out(od.ctypes.data, dc.value, 0, oi.ctypes.data, ic.value, 0, ob.ctypes.data, bc.value, 0, 0)
        res = (JobResult * max(1, n))()
        self._check(lib().dbeel_compact_many(self._h, arr, n, bloom_min_size, fp, C.byref(out), res), "dbeel_compact_many")
        return [(od[r.data_off:r.data_off + r.data_len], oi[r.index_off:r.index_off + r.index_len],
                 ob[r.bloom_off:r.bloom_off + r.bloom_len] if r.bloom_len else None, int(r.items_written)) for r in res[:n]]

    def compact_many_device(self, jobs_ptrs, out_ptrs: Tuple[int, int, int, int, int, int],
                            bloom_min_size: int = DEFAULT_BLOOM_MIN_SIZE, seeds=None, fp: float = DEFAULT_BLOOM_FP):
        """Device pointers everywhere.  Returns the JobResult rows as dicts."""
        arr, keep = self._jobs_array(jobs_ptrs, seeds)
        n = len(jobs_ptrs)
        dp, dc, ip, ic, bp, bc = out_ptrs
        out = Out(dp, dc, 0, ip, ic, 0, bp if bc else None, bc, 0, 0)
        res = (JobResult * max(1, n))()
        self._check(lib().dbeel_compact_many_device(self._h, arr, n, bloom_min_size, fp, C.byref(out), res),
                    "dbeel_compact_many_device")
        return [{k: int(getattr(r, k)) for k, _ in JobResult._fields_} for r in res[:n]]

    # ---- N4: write-ahead-log replay + flush ------------------------------------------------
    def wal_flush(self, wal, capacity: int = DEFAULT_TREE_CAPACITY):
        """dbeel_wal_flush over a host buffer holding a `.memtable` file: returns (data, index, items_written)."""
        w = _u8(wal)
        od = np.empty(max(1, w.size), np.uint8)
        oi = np.empty(max(16, (w.size + 4095) // 4096 * 16), np.uint8)
        out = Out(od.ctypes.data, od.size, 0, oi.ctypes.data, oi.size, 0, None, 0, 0, 0)
        self._check(lib().dbeel_wal_flush(self._h, w.ctypes.data if w.size else None, w.size, capacity, C.byref(out)),
                    "dbeel_wal_flush")
        return od[:out.data_len], oi[:out.index_len], int(out.items_written)

    def wal_flush_device(self, wal_ptr: int, wal_len: int, out_ptrs: Tuple[int, int, int, int],
                         capacity: int = DEFAULT_TREE_CAPACITY):
        dp, dc, ip, ic = out_ptrs
        out = Out(dp, dc, 0, ip, ic, 0, None, 0, 0, 0)
        self._check(lib().dbeel_wal_flush_device(self._h, wal_ptr, wal_len, capacity, C.byref(out)), "dbeel_wal_flush_device")
        return int(out.data_len), int(out.index_len), int(out.items_written)

    # ---- N2: batched point lookups -------------------------------------------------------
    def get_many(self, tables: Sequence[Tuple[object, object, object]], keys: Sequence[bytes],
                 mode: int = LOOKUP_REFERENCE) -> np.ndarray:
        """dbeel_get_many over host buffers.  tables: (data, index, bloom | None) oldest first, like
        LSMTree.sstables.  Returns a structured array (table, bloom_rejects, record), one row per key."""
        keep = [(_u8(d), _u8(i), _u8(b) if b is not None and len(b) else None) for d, i, b in tables]
        arr = (Table * max(1, len(keep)))()
        for j, (d, i, b) in enumerate(keep):
            arr[j] = Table(d.ctypes.data, d.size, i.ctypes.data, i.size, b.ctypes.data if b is not None else None,
                           b.size if b is not None else 0)
        blob, off = pack_keys(keys)
        res = np.zeros(len(keys), dtype=LOOKUP_DTYPE)
        self._check(lib().dbeel_get_many(self._h, arr, len(keep), blob.ctypes.data if blob.size else None,
                                         off.ctypes.data, len(keys), mode, res.ctypes.data), "dbeel_get_many")
        return res

    def get_many_device(self, tables: Sequence[Tuple[int, int, int, int, int, int]], keys_ptr: int, offsets_ptr: int,
                        n_keys: int, results_ptr: int, mode: int = LOOKUP_REFERENCE) -> None:
        """All pointers are device pointers; tables: (data_ptr, data_len, index_ptr, index_len, bloom_ptr, bloom_len)."""
        arr = (Table * max(1, len(tables)))()
        for j, t in enumerate(tables):
            arr[j] = Table(t[0], t[1], t[2], t[3], t[4] if t[5] else None, t[5])
        self._check(lib().dbeel_get_many_device(self._h, arr, len(tables), keys_ptr, offsets_ptr, n_keys, mode,
                                                results_ptr), "dbeel_get_many_device")

    # ---- hash-range scans (shard migration) ----------------------------------------------
    @staticmethod
    def _scan_args(ranges):
        rng = (HashRange * max(1, len(ranges)))()
        for j, (a, b) in enumerate(ranges):
            rng[j] = HashRange(a, b)
        return rng, (FlushTable * max(1, len(ranges)))(), ScanStop()

    @staticmethod
    def _scan_result(per_range, n, stop):
        rows = [{k: int(getattr(t, k)) for k, _ in FlushTable._fields_} for t in per_range[:n]]
        return rows, (int(stop.table), int(stop.reason), int(stop.record))

    def scan_ranges(self, tables: Sequence[Tuple[object, object]], ranges: Sequence[Tuple[int, int]],
                    mode: int = SCAN_REFERENCE, caps: Optional[Tuple[int, int]] = None):
        """dbeel_scan_ranges over host buffers.  tables: (data, index) in iteration order (SSTables oldest first, then
        the memtables as sorted runs); ranges: (start, end) hash ranges.  Returns (data, index, per_range, stop):
        per_range rows carry the dbeel_flush_table fields, stop = (table | -1, reason, record).  caps: (data_cap,
        index_cap), default the bound that always suffices."""
        keep = [(_u8(d), _u8(i)) for d, i in tables]
        arr = (Run * max(1, len(keep)))()
        for j, (d, i) in enumerate(keep):
            arr[j] = Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
        dc, ic = caps if caps is not None else (sum(d.size for d, _ in keep), 16 * sum(i.size // 16 for _, i in keep))
        od, oi = np.empty(max(1, dc), np.uint8), np.empty(max(1, ic), np.uint8)
        out = Out(od.ctypes.data, dc, 0, oi.ctypes.data, ic, 0, None, 0, 0, 0)
        rng, per_range, stop = self._scan_args(ranges)
        self._check(lib().dbeel_scan_ranges(self._h, arr, len(keep), rng, len(ranges), mode, C.byref(out), per_range,
                                            C.byref(stop)), "dbeel_scan_ranges")
        rows, st = self._scan_result(per_range, len(ranges), stop)
        return od[:out.data_len], oi[:out.index_len], rows, st

    def scan_ranges_stream(self, tables: Sequence[Tuple[object, object]], ranges: Sequence[Tuple[int, int]],
                           mode: int = SCAN_REFERENCE, partition_bytes: int = 0, read_hook=None, write_hook=None):
        """dbeel_scan_ranges_stream with in-memory "files": the engine pulls the tables through a read callback and pushes
        every range's stream through a write callback (both called from several engine threads).  Returns (data, index,
        per_range, stop) like scan_ranges(): the range streams concatenated in range order, per_range rebased to that
        concatenation.  read_hook(table, kind, offset, len) / write_hook(range, kind, offset, len), when given, run before
        every call; a nonzero return is what the callback returns (tests)."""
        import threading
        keep = [(_u8(d), _u8(i)) for d, i in tables]
        arr = (Run * max(1, len(keep)))()
        for j, (d, i) in enumerate(keep):
            arr[j] = Run(None, d.size, None, i.size)
        streams = {}  # (range, kind) -> bytearray
        mu = threading.Lock()

        def rd(_ctx, table, kind, off, n, dst):
            if read_hook is not None:
                rc = read_hook(table, kind, off, n)
                if rc:
                    return rc
            src = keep[table][0] if kind == 1 else keep[table][1]
            if off + n > src.size:
                return 4243
            C.memmove(dst, src.ctypes.data + off, n)
            return 0

        def wr(_ctx, rng_, kind, off, src, n):
            if write_hook is not None:
                rc = write_hook(rng_, kind, off, n)
                if rc:
                    return rc
            if kind not in (1, 2) or rng_ >= len(ranges):
                return 4244
            b = C.string_at(src, n)
            with mu:
                buf = streams.setdefault((rng_, kind), bytearray())
                if len(buf) < off + n:
                    buf.extend(bytes(off + n - len(buf)))
                buf[off:off + n] = b
            return 0

        io = ScanIO(SCAN_READ_FN(rd), SCAN_WRITE_FN(wr), None)
        rng, per_range, stop = self._scan_args(ranges)
        self._check(lib().dbeel_scan_ranges_stream(self._h, arr, len(keep), rng, len(ranges), mode, C.byref(io), partition_bytes,
                                                   per_range, C.byref(stop)), "dbeel_scan_ranges_stream")
        rows, st = self._scan_result(per_range, len(ranges), stop)
        data, index = bytearray(), bytearray()
        for r, row in enumerate(rows):
            d, i = bytes(streams.get((r, 1), b"")), bytes(streams.get((r, 2), b""))
            if len(d) != row["data_len"] or len(i) != row["index_len"] or row["data_off"] or row["index_off"]:
                raise AssertionError(f"range {r}: stream of {len(d)} / {len(i)} bytes against per_range {row}")
            row["data_off"], row["index_off"] = len(data), len(index)
            data += d
            index += i
        return np.frombuffer(bytes(data), np.uint8), np.frombuffer(bytes(index), np.uint8), rows, st

    def scan_ranges_device(self, tables: Sequence[Tuple[int, int, int, int]], ranges: Sequence[Tuple[int, int]],
                           out_ptrs: Tuple[int, int, int, int], mode: int = SCAN_REFERENCE):
        """dbeel_scan_ranges_device: tables (data_ptr, data_len, index_ptr, index_len) and out_ptrs (data_ptr, data_cap,
        index_ptr, index_cap) in device memory.  Returns (data_len, index_len, per_range, stop)."""
        arr = (Run * max(1, len(tables)))()
        for j, (dp, dl, ip, il) in enumerate(tables):
            arr[j] = Run(dp, dl, ip, il)
        dp, dc, ip, ic = out_ptrs
        out = Out(dp, dc, 0, ip, ic, 0, None, 0, 0, 0)
        rng, per_range, stop = self._scan_args(ranges)
        self._check(lib().dbeel_scan_ranges_device(self._h, arr, len(tables), rng, len(ranges), mode, C.byref(out),
                                                   per_range, C.byref(stop)), "dbeel_scan_ranges_device")
        rows, st = self._scan_result(per_range, len(ranges), stop)
        return int(out.data_len), int(out.index_len), rows, st

    # ---- device buffers (raw pointers; torch tensors own the memory) -------------------
    def compact_device(self, runs: Sequence[Tuple[int, int, int, int]], out_ptrs: Tuple[int, int, int, int, int, int],
                       opts: Opts) -> Tuple[int, int, int, int]:
        """runs: (data_ptr, data_len, index_ptr, index_len); out_ptrs: (data_ptr, data_cap,
        index_ptr, index_cap, bloom_ptr, bloom_cap).  Returns (data_len, index_len, bloom_len, items)."""
        arr = (Run * max(1, len(runs)))()
        for j, (dp, dl, ip, il) in enumerate(runs):
            arr[j] = Run(dp, dl, ip, il)
        dp, dc, ip, ic, bp, bc = out_ptrs
        out = Out(dp, dc, 0, ip, ic, 0, bp if bc else None, bc, 0, 0)
        self._check(lib().dbeel_compact_device(self._h, arr, len(runs), C.byref(opts), C.byref(out)),
                    "dbeel_compact_device")
        return int(out.data_len), int(out.index_len), int(out.bloom_len), int(out.items_written)

    def flush_device(self, batch: Tuple[int, int, int, int], out_ptrs: Tuple[int, int, int, int]):
        run = Run(*batch)
        dp, dc, ip, ic = out_ptrs
        out = Out(dp, dc, 0, ip, ic, 0, None, 0, 0, 0)
        self._check(lib().dbeel_flush_device(self._h, C.byref(run), C.byref(out)), "dbeel_flush_device")
        return int(out.data_len), int(out.index_len), int(out.items_written)


def murmur3_32(data: bytes, seed: int = 0) -> int:
    return int(lib().dbeel_murmur3_32(bytes(data), len(data), seed))


def shard_ring(n_shards: int, node: Optional[str] = None):
    """(ascending ring hashes, cpu id at each ring position) of a node's shards (shards.rs:213-214,657-670)."""
    h = np.zeros(n_shards, np.uint32)
    ids = np.zeros(n_shards, np.uint32)
    rc = lib().dbeel_shard_ring(node.encode() if node else None, n_shards, h.ctypes.data, ids.ctypes.data)
    if rc:
        raise DbeelError(rc, "dbeel_shard_ring")
    return h, ids


def ring_owner(ring: np.ndarray, key_hash: int) -> int:
    ring = np.ascontiguousarray(ring, np.uint32)
    return int(lib().dbeel_ring_owner(ring.ctypes.data, ring.size, key_hash))


def bind_to_gpu(device: int):
    """dbeel_bind_to_gpu: (numa node, cpus) the calling thread was bound to, (-1, 0) when there is no NUMA topology."""
    node, cpus = C.c_int(-1), C.c_int(0)
    rc = lib().dbeel_bind_to_gpu(device, C.byref(node), C.byref(cpus))
    if rc:
        raise DbeelError(rc, "dbeel_bind_to_gpu")
    return node.value, cpus.value
