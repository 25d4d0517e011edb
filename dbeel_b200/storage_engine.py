"""Python face of the host-side mirror (include/dbeel_tree.h, csrc/host/lsm_tree_host.cc).

Names and argument meaning follow the reference's storage engine so the tests read like its own
(src/storage_engine/lsm_tree.rs): ``LSMTree.open_or_create``, ``.compact(indices_to_compact,
output_index, keep_tombstones)``, ``.flush``, ``.sstable_indices_and_sizes``; the size-tiered
picker of src/tasks/compaction.rs:35-102 is ``plan_compactions`` / ``compact_tree``.
All the work happens in the C++/CUDA library; this file only marshals arguments.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import capi

ERR_IO = 20
ERR_NO_SSTABLE = 21
DEFAULT_TREE_CAPACITY = 8192  # mod.rs:18
DEFAULT_SSTABLE_BLOOM_MIN_SIZE = 1_048_576  # mod.rs:19

FILE_DATA, FILE_INDEX = 1, 2  # FileTypeKind::{Data, Index} (mod.rs:36-42)
PAGE_SIZE = 4096  # page_cache.rs:10
PAGE_SINK = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint8))

_bound = False


def _lib():
    global _bound
    L = capi.lib()
    if not _bound:
        L.dbeel_tree_open.restype = C.c_int
        L.dbeel_tree_open.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        L.dbeel_tree_close.restype = None
        L.dbeel_tree_close.argtypes = [C.c_void_p]
        L.dbeel_tree_sstables.restype = C.c_uint32
        L.dbeel_tree_sstables.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_uint32]
        L.dbeel_tree_write_sstable_index.restype = C.c_uint64
        L.dbeel_tree_write_sstable_index.argtypes = [C.c_void_p]
        L.dbeel_tree_compact.restype = C.c_int
        L.dbeel_tree_compact.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_uint64, C.c_int, C.c_char_p]
        L.dbeel_tree_flush.restype = C.c_int
        L.dbeel_tree_flush.argtypes = [C.c_void_p, C.POINTER(capi.Run), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.dbeel_tree_compact_many.restype = C.c_int
        L.dbeel_tree_compact_many.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.c_uint32,
                                              C.POINTER(C.c_uint64), C.POINTER(C.c_int32), C.c_char_p]
        L.dbeel_tree_get_many.restype = C.c_int
        L.dbeel_tree_get_many.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
        L.dbeel_tree_scan_ranges.restype = C.c_int
        L.dbeel_tree_scan_ranges.argtypes = [C.c_void_p, C.POINTER(capi.Run), C.c_uint32, C.POINTER(capi.HashRange), C.c_uint32,
                                             C.c_uint32, C.POINTER(capi.Out), C.POINTER(capi.FlushTable), C.POINTER(capi.ScanStop)]
        L.dbeel_tree_scan_ranges_to_dir.restype = C.c_int
        L.dbeel_tree_scan_ranges_to_dir.argtypes = [C.c_void_p, C.POINTER(capi.Run), C.c_uint32, C.POINTER(capi.HashRange), C.c_uint32,
                                                    C.c_uint32, C.c_char_p, C.POINTER(capi.FlushTable), C.POINTER(capi.ScanStop)]
        L.dbeel_tree_recover_wal.restype = C.c_int
        L.dbeel_tree_recover_wal.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.dbeel_tree_last_error.restype = C.c_char_p
        L.dbeel_tree_last_error.argtypes = [C.c_void_p]
        L.dbeel_memtable_cut.restype = C.c_uint64
        L.dbeel_memtable_cut.argtypes = [C.POINTER(capi.Run), C.c_uint64, C.c_uint32]
        L.dbeel_plan_compactions.restype = C.c_uint32
        L.dbeel_plan_compactions.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_uint32, C.c_uint32,
                                             C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64),
                                             C.POINTER(C.c_int32)]
        L.dbeel_out_pages.restype = C.c_int
        L.dbeel_out_pages.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint64, PAGE_SINK, C.c_void_p]
        L.dbeel_tree_set_page_sink.restype = None
        L.dbeel_tree_set_page_sink.argtypes = [C.c_void_p, PAGE_SINK, C.c_void_p]
        _bound = True
    return L


TREE_EXPORTS = ["dbeel_tree_open", "dbeel_tree_close", "dbeel_tree_sstables", "dbeel_tree_write_sstable_index",
                "dbeel_tree_compact", "dbeel_tree_compact_many", "dbeel_tree_flush", "dbeel_tree_recover_wal", "dbeel_tree_get_many", "dbeel_tree_scan_ranges", "dbeel_tree_scan_ranges_to_dir", "dbeel_tree_last_error", "dbeel_memtable_cut",
                "dbeel_plan_compactions", "dbeel_out_pages", "dbeel_tree_set_page_sink"]


def _run_struct(batch) -> Tuple[capi.Run, tuple]:
    d, i = capi._u8(batch[0]), capi._u8(batch[1])
    return capi.Run(d.ctypes.data, d.size, i.ctypes.data, i.size), (d, i)


def memtable_cut(batch, first_record: int = 0, capacity: int = DEFAULT_TREE_CAPACITY) -> int:
    """Arrivals from `first_record` on that one memtable of `capacity` distinct keys absorbs."""
    run, _keep = _run_struct(batch)
    return int(_lib().dbeel_memtable_cut(C.byref(run), first_record, capacity))


def plan_compactions(indices_and_sizes: Sequence[Tuple[int, int]], compaction_factor: int = 2):
    """compact_tree's picker, deterministic: [(indices_to_compact, output_index, keep_tombstones)]."""
    n = len(indices_and_sizes)
    if n == 0:
        return []
    idx = (C.c_uint64 * n)(*[i for i, _ in indices_and_sizes])
    siz = (C.c_uint64 * n)(*[s for _, s in indices_and_sizes])
    members = (C.c_uint64 * n)()
    start = (C.c_uint32 * (n + 1))()
    outs = (C.c_uint64 * n)()
    keeps = (C.c_int32 * n)()
    g = _lib().dbeel_plan_compactions(idx, siz, n, compaction_factor, members, start, outs, keeps)
    return [([int(members[k]) for k in range(start[j], start[j + 1])], int(outs[j]), bool(keeps[j])) for j in range(g)]


class LSMTree:
    """The compaction-facing part of dbeel's LSMTree over a directory of SSTable files."""

    def __init__(self, directory: str, engine, sstable_bloom_min_size: int = DEFAULT_SSTABLE_BLOOM_MIN_SIZE):
        self._h = C.c_void_p()
        self._engine = engine
        eh = engine._h if hasattr(engine, "_h") else engine
        rc = _lib().dbeel_tree_open(directory.encode(), eh, sstable_bloom_min_size, C.byref(self._h))
        if rc:
            raise capi.DbeelError(rc, f"dbeel_tree_open({directory})")
        self.dir = directory

    open_or_create = classmethod(lambda cls, *a, **k: cls(*a, **k))

    def close(self):
        if self._h:
            _lib().dbeel_tree_close(self._h)
            self._h = C.c_void_p()

    def set_page_cache(self, cache: Optional[dict]):
        """Mirror EntryWriter's write-through: every SSTable this tree writes from now on is also `set` page by page into
        `cache` under the reference's key ((FileTypeKind, files_index), address) (entry_writer.rs:100-156).  None = off."""
        if cache is None:
            self._sink = PAGE_SINK(0)
        else:
            def sink(_ctx, kind, files_index, address, page):
                cache[((int(kind), int(files_index)), int(address))] = bytes(page[:PAGE_SIZE])
            self._sink = PAGE_SINK(sink)
        _lib().dbeel_tree_set_page_sink(self._h, self._sink, None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc:
            raise capi.DbeelError(rc, f"{what}: {_lib().dbeel_tree_last_error(self._h).decode()}")

    def sstable_indices_and_sizes(self) -> List[Tuple[int, int]]:
        n = _lib().dbeel_tree_sstables(self._h, None, None, 0)
        idx, siz = (C.c_uint64 * max(1, n))(), (C.c_uint64 * max(1, n))()
        _lib().dbeel_tree_sstables(self._h, idx, siz, n)
        return [(int(idx[k]), int(siz[k])) for k in range(n)]

    @property
    def write_sstable_index(self) -> int:
        return int(_lib().dbeel_tree_write_sstable_index(self._h))

    def compact(self, indices_to_compact: Sequence[int], output_index: int, keep_tombstones: bool,
                bloom_seed: Optional[bytes] = None) -> None:
        arr = (C.c_uint64 * max(1, len(indices_to_compact)))(*indices_to_compact)
        self._check(_lib().dbeel_tree_compact(self._h, arr, len(indices_to_compact), output_index,
                                              int(keep_tombstones), bloom_seed), "LSMTree.compact")

    def flush(self, batch) -> Tuple[int, int]:
        """One memtable's arrivals -> the next even-indexed SSTable.  Returns (index, items)."""
        run, _keep = _run_struct(batch)
        wi, n = C.c_uint64(), C.c_uint64()
        self._check(_lib().dbeel_tree_flush(self._h, C.byref(run), C.byref(wi), C.byref(n)), "LSMTree.flush")
        return int(wi.value), int(n.value)

    def get_many(self, keys: Sequence[bytes], mode: int = capi.LOOKUP_REFERENCE):
        """get_entry's SSTable loop for a batch of keys: a list of `data` bytes (b"" = tombstone) or None per key,
        like LSMTree::get (lsm_tree.rs:722-724) after the memtables missed."""
        import numpy as np
        from . import sstable
        blob, off = capi.pack_keys(keys)
        res = np.zeros(len(keys), dtype=capi.LOOKUP_DTYPE)
        self._check(_lib().dbeel_tree_get_many(self._h, blob.ctypes.data if blob.size else None, off.ctypes.data, len(keys), mode,
                                               res.ctypes.data), "LSMTree.get_many")
        tables = self.sstable_indices_and_sizes()
        files = {}
        out = []
        for row in res:
            if row["table"] < 0:
                out.append(None)
                continue
            idx = tables[int(row["table"])][0]
            if idx not in files:
                files[idx] = sstable.read_run_files(self.dir, idx)
            d, i = files[idx]
            rec = bytes(i[16 * int(row["record"]):16 * int(row["record"]) + 16])
            o, ks, fs = int.from_bytes(rec[:8], "little"), int.from_bytes(rec[8:12], "little"), int.from_bytes(rec[12:], "little")
            out.append(bytes(d[o + ks + 8:o + fs - 16]))  # EntryValue.data (entry = key | dlen | data | ts)
        return out

    def scan_ranges(self, ranges: Sequence[Tuple[int, int]], mode: int = capi.SCAN_REFERENCE, memtables=()):
        """The scan of migrate_actions (migration.rs:62-131) over this tree: every entry whose murmur3_32(key) lies in
        one of `ranges`, assigned to the first range that holds.  memtables: (data, index) sorted runs of the flushing
        and then the active memtable.  Returns (data, index, per_range, stop) like capi.Engine.scan_ranges, stop's table
        counting the SSTables in sstable_indices_and_sizes() order and then `memtables`."""
        from . import sstable
        keep = [(capi._u8(d), capi._u8(i)) for d, i in memtables]
        mts = (capi.Run * max(1, len(keep)))()
        for j, (d, i) in enumerate(keep):
            mts[j] = capi.Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
        dc = sum(d.size for d, _ in keep)
        ic = 16 * sum(i.size // 16 for _, i in keep)
        for idx, size in self.sstable_indices_and_sizes():
            d, i = sstable.read_run_files(self.dir, idx)
            dc += len(d)
            ic += 16 * (len(i) // 16)
        od, oi = np.empty(max(1, dc), np.uint8), np.empty(max(1, ic), np.uint8)
        out = capi.Out(od.ctypes.data, dc, 0, oi.ctypes.data, ic, 0, None, 0, 0, 0)
        rng, per_range, stop = capi.Engine._scan_args(ranges)
        self._check(_lib().dbeel_tree_scan_ranges(self._h, mts, len(keep), rng, len(ranges), mode, C.byref(out), per_range,
                                                  C.byref(stop)), "LSMTree.scan_ranges")
        rows, st = capi.Engine._scan_result(per_range, len(ranges), stop)
        return od[:out.data_len], oi[:out.index_len], rows, st

    def scan_ranges_to_dir(self, ranges: Sequence[Tuple[int, int]], out_dir: str, mode: int = capi.SCAN_REFERENCE,
                           memtables=()):
        """scan_ranges streamed from the tree's files: range r goes to <out_dir>/<r>.data and <out_dir>/<r>.index
        (dbeel_tree_scan_ranges_to_dir).  Returns (per_range, stop): per_range rows with data_off == index_off == 0, stop
        as in scan_ranges."""
        keep = [(capi._u8(d), capi._u8(i)) for d, i in memtables]
        mts = (capi.Run * max(1, len(keep)))()
        for j, (d, i) in enumerate(keep):
            mts[j] = capi.Run(d.ctypes.data, d.size, i.ctypes.data, i.size)
        rng, per_range, stop = capi.Engine._scan_args(ranges)
        self._check(_lib().dbeel_tree_scan_ranges_to_dir(self._h, mts, len(keep), rng, len(ranges), mode, os.fsencode(out_dir),
                                                         per_range, C.byref(stop)), "LSMTree.scan_ranges_to_dir")
        return capi.Engine._scan_result(per_range, len(ranges), stop)

    def recover_wal(self, tree_capacity: int = capi.DEFAULT_TREE_CAPACITY) -> Tuple[int, int]:
        """open_or_create_ex's WAL step (lsm_tree.rs:466-513): with two `.memtable` files the older one is replayed and
        flushed.  Returns (index of the log that stays active, entries of the recovered SSTable)."""
        wi, n = C.c_uint64(), C.c_uint64()
        self._check(_lib().dbeel_tree_recover_wal(self._h, tree_capacity, C.byref(wi), C.byref(n)), "LSMTree.recover_wal")
        return int(wi.value), int(n.value)

    def compact_many(self, plan, bloom_seeds: Optional[Sequence[bytes]] = None) -> None:
        """All groups of a plan_compactions() result through ONE dbeel_compact_many, committed group by group."""
        members = [i for indices, _, _ in plan for i in indices]
        starts = [0]
        for indices, _, _ in plan:
            starts.append(starts[-1] + len(indices))
        n = len(plan)
        m = (C.c_uint64 * max(1, len(members)))(*members)
        gs = (C.c_uint32 * (n + 1))(*starts)
        oi = (C.c_uint64 * max(1, n))(*[o for _, o, _ in plan])
        kt = (C.c_int32 * max(1, n))(*[int(k) for _, _, k in plan])
        seeds = b"".join(bloom_seeds) if bloom_seeds is not None else None
        self._check(_lib().dbeel_tree_compact_many(self._h, m, gs, n, oi, kt, seeds), "LSMTree.compact_many")

    def compact_tree(self, compaction_factor: int = 2, bloom_seed: Optional[bytes] = None, batched: bool = False):
        """tasks/compaction.rs compact_tree: plan with the picker, run every group (batched: in one launch sequence)."""
        plan = plan_compactions(self.sstable_indices_and_sizes(), compaction_factor)
        if batched and plan:
            self.compact_many(plan, [bloom_seed] * len(plan) if bloom_seed is not None else None)
            return plan
        for indices, out, keep in plan:
            self.compact(indices, out, keep, bloom_seed)
        return plan


def out_pages(data, index, files_index: int):
    """dbeel_out_pages: the (file kind, files_index, address, page bytes) sequence EntryWriter would `set` for this SSTable."""
    d, i = capi._u8(data), capi._u8(index)
    seq = []

    def sink(_ctx, kind, fi, address, page):
        seq.append((int(kind), int(fi), int(address), bytes(page[:PAGE_SIZE])))
    cb = PAGE_SINK(sink)
    rc = _lib().dbeel_out_pages(d.ctypes.data if d.size else None, d.size, i.ctypes.data if i.size else None, i.size, files_index, cb, None)
    if rc:
        raise capi.DbeelError(rc, "dbeel_out_pages")
    return seq
