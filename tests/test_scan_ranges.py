"""Hash-range scans (dbeel_scan_ranges): the scan of migrate_actions (src/tasks/migration.rs:62-131) over
LSMTree::iter_filter (src/storage_engine/lsm_tree.rs:133-282).

CPU: the scan oracle against the reference's own iterator test and against a literal Python restatement of read_one +
migrate_actions; the device-side predicates (device_fns.cuh, built by g++) against the same restatement.
GPU: every case byte-compared with the oracle -- every range's .data / .index, per_range and the stop."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import oracle
import scan_oracle
from dbeel_b200 import sstable
from dbeel_b200 import workloads as W
from helpers import BASE_TS, nasty_keys

HERE = os.path.dirname(os.path.abspath(__file__))
REF, EXACT = scan_oracle.SCAN_REFERENCE, scan_oracle.SCAN_EXACT
END, DECODE, READ = scan_oracle.SCAN_END, scan_oracle.SCAN_DECODE, scan_oracle.SCAN_READ
ALL = [(1, 0)]  # wrapped: in REFERENCE mode it holds for every hash


# ----------------------------------------------------------------------------- literal restatement

def between_cmp(h, start, end, mode=REF):
    """migration.rs:54-60; mode EXACT reads a wrapped range as [start, 2^32) u [0, end)."""
    if end < start:
        return (h >= start or h < end) if mode == EXACT else (h < start or h >= end)
    return start <= h < end


def decode_entry(b: bytes):
    """bincode Entry from exactly len(b) bytes (reject_trailing_bytes) + the timestamp range: (key, data) or None."""
    n = len(b)
    if n < 8:
        return None
    klen = int.from_bytes(b[:8], "little")
    if klen > n - 8 or n - 8 - klen < 8:
        return None
    dlen = int.from_bytes(b[8 + klen:16 + klen], "little")
    if dlen > n - 16 - klen or n - 16 - klen - dlen != 16:
        return None
    if not oracle.timestamp_decodes(int.from_bytes(b[n - 16:], "little", signed=True)):
        return None
    return b[8:8 + klen], b[16 + klen:16 + klen + dlen]


def py_scan(tables, ranges, mode=REF):
    """AsyncIter::read_one + migrate_actions' filter and `position`: (entries per range, stop)."""
    outs = [[] for _ in ranges]
    for t, (d, i) in enumerate(tables):
        d, i = bytes(d), bytes(i)
        size = len(i) // 16
        if size == 0:
            return outs, (t, READ, 0)  # the first 16-byte index read hits EOF
        for r in range(size):
            off, _ks, fs = struct.unpack_from("<QII", i, 16 * r)
            if fs == 0 or off + fs > len(d):
                return outs, (t, READ, r)
            b = d[off:off + fs]
            ent = decode_entry(b)
            if ent is None:
                return outs, (t, DECODE, r)
            h = oracle.murmur3_32(ent[0])
            pos = next((k for k, (s, e) in enumerate(ranges) if between_cmp(h, s, e, mode)), None)
            if pos is not None:
                outs[pos].append((b, len(ent[0])))
    return outs, (-1, END, 0)


def expected_outputs(outs):
    """Range-major .data / .index with every range's offsets relative to its own start."""
    d, i, rows = bytearray(), bytearray(), []
    for ents in outs:
        d0, i0, off = len(d), len(i), 0
        for b, klen in ents:
            i += struct.pack("<QII", off, 8 + klen, len(b))
            d += b
            off += len(b)
        rows.append(dict(data_off=d0, data_len=len(d) - d0, index_off=i0, index_len=len(i) - i0, items=len(ents)))
    return bytes(d), bytes(i), rows


def check_oracle_matches_model(tables, ranges, mode):
    od, oi, rows, stop = scan_oracle.scan_ranges(tables, ranges, mode)
    outs, mstop = py_scan(tables, ranges, mode)
    ed, ei, erows = expected_outputs(outs)
    assert stop == mstop
    assert rows == erows
    assert bytes(od) == ed and bytes(oi) == ei
    return od, oi, rows, stop


# ----------------------------------------------------------------------------- trees

def u16key(n):
    return int(n).to_bytes(2, "little")


def sorted_run(entries):
    return sstable.build_run(sorted(entries, key=lambda e: e[0]))


def random_tree(rng, n_tables, per_table, n_mem=1):
    """SSTables over a shared nasty key pool (repeated versions, tombstones), then sorted memtable runs."""
    pool = nasty_keys(rng, max(8, per_table * 2), max_len=90)
    tables = []
    for t in range(n_tables + n_mem):
        n = int(rng.integers(1, per_table + 1))
        keys = sorted(pool[j] for j in rng.choice(len(pool), size=min(n, len(pool)), replace=False))
        ents = [(k, b"" if rng.random() < 0.2 else bytes(rng.integers(0, 256, int(rng.integers(1, 70)), dtype=np.uint8)),
                 BASE_TS + int(rng.integers(-99, 99))) for k in keys]
        tables.append(sstable.build_run(ents))
    return tables


def damage(rng, tables, kind):
    """One record (or table) the iterator cannot yield, at a random position."""
    tables = [(d.copy(), i.copy()) for d, i in tables]
    t = int(rng.integers(len(tables)))
    if kind == "empty":
        tables.insert(t, (np.zeros(0, np.uint8), np.zeros(0, np.uint8)))
        return tables
    d, i = tables[t]
    r = int(rng.integers(i.size // 16))
    off, ks, fs = struct.unpack_from("<QII", i.tobytes(), 16 * r)
    if kind == "decode":  # key length prefix past the entry
        d[off:off + 8] = np.frombuffer(struct.pack("<Q", fs), np.uint8)
    elif kind == "timestamp":  # year > 9999
        d[off + fs - 16:off + fs] = np.frombuffer((1 << 100).to_bytes(16, "little", signed=True), np.uint8)
    elif kind == "zero":
        i[16 * r + 12:16 * r + 16] = 0
    elif kind == "eof":
        i[16 * r:16 * r + 8] = np.frombuffer(struct.pack("<Q", d.size - fs + 1), np.uint8)
    return tables


DAMAGES = ["decode", "timestamp", "zero", "eof", "empty"]


# ----------------------------------------------------------------------------- CPU: the reference's own test

def _values_in(tables, lo, hi):
    od, oi, rows, stop = scan_oracle.scan_ranges(tables, ALL, REF)
    assert stop == (-1, END, 0)
    return [v for k, v, _ in sstable.parse_run(od, oi) if lo <= k < hi]


def test_oracle_reproduces_get_after_compaction_iter():
    """lsm_tree.rs:1332-1397: iter_filter([1,0] <= k < [5,0]) before the deletes, after them (before and after the
    manual flush) and after compact(&[0, 2, 4], 5, false)."""
    writes = [(u16key(n), u16key(n), BASE_TS + n) for n in range(32 * 3 - 2)]
    deletes = [(u16key(1), b"", BASE_TS + 1000), (u16key(4), b"", BASE_TS + 1001)]
    flushed = oracle.memtable_flushes(sstable.build_run(writes + deletes), capacity=32)
    assert [n for _, _, n in flushed] == [32, 32, 32]
    t0, t2, t4 = [(d, i) for d, i, _ in flushed]
    lo, hi = u16key(1), u16key(5)
    active = sorted_run(writes[64:])  # two automatic flushes, 30 keys still in the memtable
    assert _values_in([t0, t2, active], lo, hi) == [u16key(1), u16key(2), u16key(3), u16key(4)]
    post = [u16key(1), u16key(2), u16key(3), u16key(4), b"", b""]
    assert _values_in([t0, t2, sorted_run(writes[64:] + deletes)], lo, hi) == post  # the full memtable, before the flush
    assert _values_in([t0, t2, t4], lo, hi) == post  # ... and flushed to table 4
    d, i, _, n = oracle.compact([t0, t2, t4], keep_tombstones=False)
    assert n == 92
    assert _values_in([(d, i)], lo, hi) == [u16key(2), u16key(3)]


# ----------------------------------------------------------------------------- CPU: oracle vs restatement

@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_restatement_on_random_trees(seed):
    rng = np.random.default_rng(100 + seed)
    tables = random_tree(rng, int(rng.integers(1, 6)), 40, n_mem=int(rng.integers(0, 3)))
    for mode in (REF, EXACT):
        cuts = np.sort(rng.integers(0, 1 << 32, 4, dtype=np.uint64)).astype(int)
        ranges = [(cuts[0], cuts[1]), (cuts[3], cuts[2]), (cuts[1], cuts[3]), (7, 7)]  # one wrapped, one empty
        check_oracle_matches_model(tables, ranges, mode)
        check_oracle_matches_model(tables, ALL, mode)
        check_oracle_matches_model(tables, [], mode)


@pytest.mark.parametrize("kind", DAMAGES)
def test_oracle_stops_like_the_restatement(kind):
    rng = np.random.default_rng(50 + DAMAGES.index(kind))
    for trial in range(4):
        tables = damage(rng, random_tree(rng, 4, 30), kind)
        _, _, _, stop = check_oracle_matches_model(tables, [(0, 1 << 31), (5, 3)], REF)
        assert stop[1] == (DECODE if kind in ("decode", "timestamp") else READ)


# ----------------------------------------------------------------------------- CPU: device predicates under g++

@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "scan_shim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", so,
                           os.path.join(HERE, "scan_shim.cc")])
    L = C.CDLL(so)
    L.shim_hash_in_range.restype = C.c_int
    L.shim_hash_in_range.argtypes = [C.c_uint32] * 4
    L.shim_entry_readable.restype = C.c_int
    L.shim_entry_readable.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64]
    L.shim_entry_decodes.restype = C.c_int
    L.shim_entry_decodes.argtypes = [C.c_char_p, C.c_uint64]
    return L


def test_hash_in_range_every_boundary(shim):
    M = (1 << 32) - 1
    pts = [0, 1, 2, 1 << 31, M - 1, M]
    for s in pts:
        for e in pts:
            for h in sorted(set(pts + [(s + 1) & M, (s - 1) & M, (e + 1) & M, (e - 1) & M])):
                for mode in (REF, EXACT):
                    want = between_cmp(h, s, e, mode)
                    assert bool(shim.shim_hash_in_range(h, s, e, mode)) == want, (h, s, e, mode)
                    assert scan_oracle.between_cmp(h, s, e, mode) == want, (h, s, e, mode)
    assert all(shim.shim_hash_in_range(h, 9, 3, REF) for h in (0, 3, 5, 9, M))  # wrapped, literal: everything
    assert not any(shim.shim_hash_in_range(h, 5, 5, m) for h in (0, 4, 5, 6, M) for m in (REF, EXACT))


def test_read_rule_every_boundary(shim):
    M64 = (1 << 64) - 1
    for off, fs, n in [(0, 0, 10), (0, 10, 10), (0, 11, 10), (10, 0, 10), (10, 1, 10), (11, 1, 10), (M64, 1, 10),
                       (5, (1 << 32) - 1, 10), (0, (1 << 32) - 1, (1 << 32) - 1), (M64 - 3, 4, M64)]:
        want = fs != 0 and off + fs <= n
        assert bool(shim.shim_entry_readable(off, fs, n)) == want, (off, fs, n)


def test_decode_rule_against_restatement(shim):
    rng = np.random.default_rng(7)
    good = sstable.encode_entry(b"key", b"value", BASE_TS)
    cases = [good, sstable.encode_entry(b"", b"", 0), sstable.encode_entry(b"k" * 70, b"", -1)]
    for ts in (-(1 << 127), (1 << 127) - 1, 253402300799 * 10**9 + 999999999, 253402300800 * 10**9,
               -377705116800 * 10**9, -377705116800 * 10**9 - 1):
        cases.append(sstable.encode_entry(b"ab", b"c", ts))
    for cut in range(len(good) + 1):
        cases.append(good[:cut])
    cases.append(good + b"\x00")
    for klen in (0, 2, 3, 4, 5, len(good) - 32, len(good) - 31, len(good) - 8, len(good), 1 << 40, (1 << 64) - 1):
        cases.append(struct.pack("<Q", klen) + good[8:])
    for dlen in (0, 4, 5, 6, 1 << 63):
        cases.append(good[:11] + struct.pack("<Q", dlen) + good[19:])
    for _ in range(200):
        b = bytearray(good)
        b[int(rng.integers(len(b)))] = int(rng.integers(256))
        cases.append(bytes(b))
    for b in cases:
        assert bool(shim.shim_entry_decodes(b, len(b))) == (decode_entry(b) is not None), b


# ----------------------------------------------------------------------------- GPU

def assert_scan_equal(got, exp, what=""):
    gd, gi, grows, gstop = got
    ed, ei, erows, estop = exp
    assert gstop == estop, f"{what}: stop {gstop} != {estop}"
    assert grows == erows, f"{what}: per_range differs"
    assert np.array_equal(np.asarray(gi), np.asarray(ei)), f"{what}: .index differs"
    assert np.array_equal(np.asarray(gd), np.asarray(ed)), f"{what}: .data differs"


def gpu_vs_oracle(engine, tables, ranges, mode=REF, what=""):
    got = engine.scan_ranges(tables, ranges, mode)
    exp = scan_oracle.scan_ranges(tables, ranges, mode)
    assert_scan_equal(got, exp, what)
    return got


def ring_ranges(n):
    """n arcs of a ring of n shards: (previous, this) -- the lowest one wraps."""
    h = sorted(oracle.murmur3_32(f"dbeel-{k}".encode()) for k in range(n))
    return [(h[k - 1], h[k]) for k in range(n)]


@pytest.fixture(scope="module")
def cfg2_runs():
    return W.make_merge_runs(W.scaled(W.CFG2, 6_000))


@pytest.mark.gpu
def test_gpu_shapes(engine, cfg2_runs):
    rng = np.random.default_rng(11)
    small = random_tree(rng, 1, 50, n_mem=0)
    gpu_vs_oracle(engine, small, [(0, 1 << 31)], REF, "1 table x 1 range")
    for n in (1, 3, 64, 256):
        for mode in (REF, EXACT):
            gpu_vs_oracle(engine, cfg2_runs, ring_ranges(n), mode, f"cfg2 x {n} ranges mode {mode}")
    ragged = random_tree(rng, 37, 60, n_mem=0)
    gpu_vs_oracle(engine, ragged, ring_ranges(5), EXACT, "37 ragged tables")
    mem = sorted_run([(b"mem-%d" % k, b"v" * (k % 9), BASE_TS + k) for k in range(500)])
    gpu_vs_oracle(engine, cfg2_runs + [mem], ring_ranges(3), EXACT, "memtable run appended")
    gpu_vs_oracle(engine, [], ring_ranges(3), EXACT, "zero tables")
    got = gpu_vs_oracle(engine, cfg2_runs, [], REF, "zero ranges")
    assert got[0].size == 0 and got[1].size == 0


@pytest.mark.gpu
def test_gpu_range_cases(engine, cfg2_runs):
    rng = np.random.default_rng(12)
    tree = random_tree(rng, 6, 300, n_mem=2)
    for mode in (REF, EXACT):
        gpu_vs_oracle(engine, tree, [(3_000_000_000, 1_000_000_000)], mode, "wrapped")
        gpu_vs_oracle(engine, tree, [(0, 2_000_000_000), (1_000_000_000, 3_000_000_000), (4_000_000_000, 500)], mode,
                      "overlapping: first match wins")
        got = gpu_vs_oracle(engine, tree, [(5, 5), (9, 9)], mode, "selects nothing")
        assert got[0].size == 0
    got = gpu_vs_oracle(engine, cfg2_runs, ALL, REF, "everything")
    assert got[3] == (-1, END, 0) and got[2][0]["items"] == sum(i.size // 16 for _, i in cfg2_runs)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", DAMAGES)
def test_gpu_stops(engine, kind):
    rng = np.random.default_rng(20 + DAMAGES.index(kind))
    for trial in range(3):
        tables = damage(rng, random_tree(rng, 5, 200, n_mem=2), kind)
        got = gpu_vs_oracle(engine, tables, ring_ranges(4) + [(1, 0)], REF, f"{kind} #{trial}")
        assert got[3][1] == (DECODE if kind in ("decode", "timestamp") else READ)


@pytest.mark.gpu
def test_gpu_stop_positions(engine, cfg2_runs):
    """A stop in table 0, in a middle table and in the last record; a stop in an SSTable drops the memtables behind it."""
    mem = sorted_run([(b"m%05d" % k, b"x", BASE_TS) for k in range(300)])
    base = [(d.copy(), i.copy()) for d, i in cfg2_runs] + [mem]
    for t, r in [(0, 0), (0, 17), (4, 1234), (7, cfg2_runs[7][1].size // 16 - 1), (8, 299)]:
        tables = [(d.copy(), i.copy()) for d, i in base]
        tables[t][1][16 * r + 12:16 * r + 16] = 0
        got = gpu_vs_oracle(engine, tables, ALL, REF, f"stop at {t}/{r}")
        assert got[3] == (t, READ, r)
        if t < 8:
            assert not any(k.startswith(b"m0") for k, _, _ in sstable.parse_run(got[0], got[1]))


@pytest.mark.gpu
def test_gpu_host_equals_device(engine, cfg2_runs):
    import torch
    ranges = ring_ranges(3)
    host = engine.scan_ranges(cfg2_runs, ranges, EXACT)
    dev = [(torch.from_numpy(d).cuda(), torch.from_numpy(i).cuda()) for d, i in cfg2_runs]
    dc, ic = sum(d.size for d, _ in cfg2_runs), sum(i.size for _, i in cfg2_runs)
    od, oi = torch.empty(dc, dtype=torch.uint8, device="cuda"), torch.empty(ic, dtype=torch.uint8, device="cuda")
    dl, il, rows, stop = engine.scan_ranges_device([(d.data_ptr(), d.numel(), i.data_ptr(), i.numel()) for d, i in dev],
                                                   ranges, (od.data_ptr(), dc, oi.data_ptr(), ic), EXACT)
    assert_scan_equal((od[:dl].cpu().numpy(), oi[:il].cpu().numpy(), rows, stop), host, "device form")


@pytest.mark.gpu
def test_gpu_capacity_then_reuse(engine, cfg2_runs):
    from dbeel_b200 import capi
    ranges = ring_ranges(2)
    _, _, rows, _ = scan_oracle.scan_ranges(cfg2_runs, ranges, EXACT)
    need_d, need_i = sum(r["data_len"] for r in rows), sum(r["index_len"] for r in rows)
    for caps in ((need_d - 1, need_i), (need_d, need_i - 1)):
        with pytest.raises(capi.DbeelError) as ex:
            engine.scan_ranges(cfg2_runs, ranges, EXACT, caps=caps)
        assert ex.value.code == capi.ERR_CAPACITY
    assert_scan_equal(engine.scan_ranges(cfg2_runs, ranges, EXACT, caps=(need_d, need_i)),
                      scan_oracle.scan_ranges(cfg2_runs, ranges, EXACT), "exact caps after a capacity error")
    with pytest.raises(capi.DbeelError) as ex:
        engine.scan_ranges(cfg2_runs, [(0, 1)] * 257, EXACT)
    assert ex.value.code == capi.ERR_INVALID_ARG


@pytest.mark.gpu
def test_gpu_every_range_flushes_like_the_oracle(engine):
    """Every range's output is an arrival batch the receiving shard can flush as is."""
    rng = np.random.default_rng(31)
    tree = random_tree(rng, 4, 400, n_mem=1)
    d, i, rows, _ = engine.scan_ranges(tree, ring_ranges(4), EXACT)
    for row in rows:
        batch = (d[row["data_off"]:row["data_off"] + row["data_len"]].copy(),
                 i[row["index_off"]:row["index_off"] + row["index_len"]].copy())
        if not row["items"]:
            continue
        t = oracle.RbTree(row["items"])
        for k, v, ts in sstable.parse_run(*batch):
            t.set(k, v, ts)
        ed, ei, _ = t.flush(cap_bytes=row["data_len"] + row["index_len"] + 4096)
        gd, gi, _ = engine.flush(batch)
        assert np.array_equal(gd, ed) and np.array_equal(gi, ei)


@pytest.mark.gpu
def test_gpu_lsm_tree_scan(engine, tmp_path):
    from dbeel_b200 import storage_engine as se
    rng = np.random.default_rng(41)
    tree = se.LSMTree(str(tmp_path), engine)
    try:
        batches = random_tree(rng, 4, 300, n_mem=0)
        for b in batches:
            tree.flush(b)
        idx = [k for k, _ in tree.sstable_indices_and_sizes()]
        tree.compact(idx[:2], idx[1] + 1, False)
        mem = sorted_run([(b"active-%d" % k, b"v", BASE_TS) for k in range(50)])
        files = [sstable.read_run_files(str(tmp_path), k) for k, _ in tree.sstable_indices_and_sizes()]
        for mode in (REF, EXACT):
            got = tree.scan_ranges(ring_ranges(3), mode, memtables=[mem])
            assert_scan_equal(got, scan_oracle.scan_ranges(files + [mem], ring_ranges(3), mode), f"LSMTree mode {mode}")
    finally:
        tree.close()
