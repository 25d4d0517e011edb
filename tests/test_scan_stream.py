"""Streamed hash-range scans (dbeel_scan_ranges_stream, LSMTree.scan_ranges_to_dir): every case byte-compared with the
whole-buffer scan (Engine.scan_ranges) and the CPU scan oracle -- every range's stream, per_range and the stop -- over
partition sizes that make partitions span tables, hold single records and leave ranges empty in some partitions."""
import os
import struct

import numpy as np
import pytest

import oracle
import scan_oracle
from dbeel_b200 import sstable
from dbeel_b200 import workloads as W
from helpers import BASE_TS
from test_scan_plan import plan as plan_of
from test_scan_plan import shim  # noqa: F401  (fixture)
from test_scan_ranges import ALL, DAMAGES, DECODE, END, EXACT, READ, REF, assert_scan_equal, random_tree, ring_ranges, sorted_run

pytestmark = pytest.mark.gpu

KIB = 1024
PARTITIONS = [4 * KIB, 64 * KIB, 1024 * KIB, 0]  # 0: the engine's partition size


def expected_lengths(exp):
    """(range, kind) -> final stream length, from a (data, index, per_range, stop) result."""
    return {**{(r, 1): row["data_len"] for r, row in enumerate(exp[2])}, **{(r, 2): row["index_len"] for r, row in enumerate(exp[2])}}


def streamed(engine, tables, ranges, mode, pb, exp=None):
    """scan_ranges_stream, with a sink that refuses any byte past the expected end of its stream."""
    exp = exp if exp is not None else scan_oracle.scan_ranges(tables, ranges, mode)
    lens = expected_lengths(exp)

    def sink(r, kind, off, n):
        return 0 if off + n <= lens[(r, kind)] and n > 0 else 99

    got = engine.scan_ranges_stream(tables, ranges, mode, pb, write_hook=sink)
    assert_scan_equal(got, exp, f"streamed, partition_bytes {pb}")
    return got, exp


@pytest.fixture(scope="module")
def cfg2_small():
    return W.make_merge_runs(W.scaled(W.CFG2, 3_000))


def test_parity_random_trees(engine):
    rng = np.random.default_rng(61)
    for trial in range(4):
        tree = random_tree(rng, int(rng.integers(1, 6)), 300, n_mem=int(rng.integers(0, 3)))
        for n in (1, 3, 17, 256):
            ranges = ring_ranges(n)
            for mode in (REF, EXACT):
                exp = scan_oracle.scan_ranges(tree, ranges, mode)
                assert_scan_equal(engine.scan_ranges(tree, ranges, mode), exp, "whole-buffer")
                for pb in PARTITIONS[:2] if n == 256 else PARTITIONS:
                    streamed(engine, tree, ranges, mode, pb, exp)
        for mode in (REF, EXACT):
            for pb in PARTITIONS:
                streamed(engine, tree, ALL, mode, pb)
                streamed(engine, tree, [], mode, pb)
                streamed(engine, [], ring_ranges(3), mode, pb)


def test_parity_cfg2_partitions_span_tables(engine, cfg2_small):
    mem = sorted_run([(b"mem-%d" % k, b"v" * (k % 9), BASE_TS + k) for k in range(500)])
    tables = cfg2_small + [mem]
    for ranges, mode in ((ring_ranges(3), EXACT), (ALL, REF), (ring_ranges(64), REF)):
        exp = engine.scan_ranges(tables, ranges, mode)
        assert_scan_equal(exp, scan_oracle.scan_ranges(tables, ranges, mode), "whole-buffer")
        for pb in (64 * KIB, 1024 * KIB, 0):
            streamed(engine, tables, ranges, mode, pb, exp)
            st = engine.stats()
            assert st["entries_out"] == sum(r["items"] for r in exp[2])
            assert st["output_bytes"] == exp[0].size + exp[1].size
            if pb:
                assert st["partitions"] > 1


def test_single_record_partitions_and_large_records(engine):
    rng = np.random.default_rng(62)
    big = sorted_run([(b"big-%d" % k, bytes(rng.integers(0, 256, 9000 + 97 * k, dtype=np.uint8)), BASE_TS) for k in range(40)])
    tables = random_tree(rng, 2, 100, n_mem=0) + [big] + random_tree(rng, 1, 100, n_mem=1)
    for pb in (1, 4 * KIB, 64 * KIB):
        streamed(engine, tables, ring_ranges(5), EXACT, pb)
        if pb == 1:
            assert engine.stats()["partitions"] == sum(i.size // 16 for _, i in tables)


def damage_at(tables, t, r, kind):
    """damage() of test_scan_ranges at a chosen record."""
    tables = [(d.copy(), i.copy()) for d, i in tables]
    if kind == "empty":
        tables.insert(t, (np.zeros(0, np.uint8), np.zeros(0, np.uint8)))
        return tables
    d, i = tables[t]
    off, ks, fs = struct.unpack_from("<QII", i.tobytes(), 16 * r)
    if kind == "decode":
        d[off:off + 8] = np.frombuffer(struct.pack("<Q", fs), np.uint8)
    elif kind == "timestamp":
        d[off + fs - 16:off + fs] = np.frombuffer((1 << 100).to_bytes(16, "little", signed=True), np.uint8)
    elif kind == "zero":
        i[16 * r + 12:16 * r + 16] = 0
    elif kind == "eof":
        i[16 * r:16 * r + 8] = np.frombuffer(struct.pack("<Q", d.size - fs + 1), np.uint8)
    return tables


@pytest.mark.parametrize("kind", DAMAGES)
def test_stops_at_partition_edges(engine, shim, kind):  # noqa: F811
    rng = np.random.default_rng(70 + DAMAGES.index(kind))
    pb = 8 * KIB
    tree = random_tree(rng, 5, 200, n_mem=2)
    pieces, parts, _, _ = plan_of(shim, tree, pb)
    assert len(parts) >= 4
    positions = []
    for c in (1, len(parts) // 2):
        mine = [p for p in pieces if p[0] == c]
        nxt = [p for p in pieces if p[0] == c + 1]
        positions += [(mine[0][1], mine[0][2]), (mine[-1][1], mine[-1][3] - 1), (nxt[0][1], nxt[0][2])]
    for _ in range(3):
        t = int(rng.integers(len(tree)))
        positions.append((t, int(rng.integers(tree[t][1].size // 16))))
    for t, r in positions:
        if kind == "empty":
            r = 0
        tables = damage_at(tree, t, r, kind)
        for mode, ranges in ((REF, ring_ranges(4) + [(1, 0)]), (EXACT, ring_ranges(3))):
            got, exp = streamed(engine, tables, ranges, mode, pb)
            assert got[3] == (t, DECODE if kind in ("decode", "timestamp") else READ, r)
            assert_scan_equal(engine.scan_ranges(tables, ranges, mode), exp, "whole-buffer")


def test_scattered_offsets(engine):
    rng = np.random.default_rng(80)
    tree = random_tree(rng, 4, 300, n_mem=1)
    scattered = []
    for d, i in tree:  # permuted readable index records within every table
        rec = i.reshape(-1, 16)
        scattered.append((d, rec[rng.permutation(len(rec))].reshape(-1).copy()))
    for pb in (4 * KIB, 64 * KIB, 0):
        for mode in (REF, EXACT):
            streamed(engine, scattered, ring_ranges(6), mode, pb)


def test_callback_errors_leave_the_engine_usable(engine, cfg2_small):
    from dbeel_b200 import capi
    ranges = ring_ranges(4)
    exp = scan_oracle.scan_ranges(cfg2_small, ranges, EXACT)
    pb = 256 * KIB

    def failing(kind_wanted, at):
        calls = {"n": 0}
        import threading
        mu = threading.Lock()

        def hook(_idx, kind, off, n):
            if kind != kind_wanted:
                return 0
            with mu:
                k = calls["n"]
                calls["n"] += 1
            return 77 if k == at else 0
        return hook

    cases = [dict(read_hook=failing(2, 0)), dict(read_hook=failing(1, 0)), dict(read_hook=failing(1, 7)),
             dict(read_hook=failing(1, 25)), dict(write_hook=failing(1, 0)), dict(write_hook=failing(2, 5)),
             dict(write_hook=failing(1, 40))]
    for hooks in cases:
        with pytest.raises(capi.DbeelError) as ex:
            engine.scan_ranges_stream(cfg2_small, ranges, EXACT, pb, **hooks)
        assert ex.value.code == 77, hooks
        streamed(engine, cfg2_small, ranges, EXACT, pb, exp)
        assert_scan_equal(engine.scan_ranges(cfg2_small, ranges, EXACT), exp, "whole-buffer after a callback error")
    gd, gi, _, gn = engine.compact(cfg2_small[:3], seed=bytes(32), bloom_min_size=1 << 40)
    od, oi, _, on = oracle.compact(cfg2_small[:3], keep_tombstones=False, seed=bytes(32), bloom_min_size=1 << 40)
    assert gn == on and np.array_equal(gd, od) and np.array_equal(gi, oi)


def test_lsm_tree_scan_to_dir(engine, tmp_path):
    from dbeel_b200 import capi
    from dbeel_b200 import storage_engine as se
    rng = np.random.default_rng(90)
    tdir = tmp_path / "tree"
    tdir.mkdir()
    tree = se.LSMTree(str(tdir), engine)
    try:
        for b in random_tree(rng, 4, 400, n_mem=0):
            tree.flush(b)
        idx = [k for k, _ in tree.sstable_indices_and_sizes()]
        tree.compact(idx[:2], idx[1] + 1, False)
    finally:
        tree.close()
    mem = sorted_run([(b"active-%d" % k, b"v" * (k % 5), BASE_TS) for k in range(300)])
    empty = (np.zeros(0, np.uint8), np.zeros(0, np.uint8))
    broken = damage_at([mem], 0, 120, "zero")[0]
    old = {k: os.environ.get(k) for k in ("DBEEL_STREAM_RING", "DBEEL_PARTITION_KB")}
    os.environ.update(DBEEL_STREAM_RING="2", DBEEL_PARTITION_KB="16")
    try:
        small = capi.Engine(0)  # ring of two slots, 16 KiB partitions
    finally:
        for k, v in old.items():
            os.environ.pop(k) if v is None else os.environ.__setitem__(k, v)
    try:
        for eng in (engine, small):
            tree = se.LSMTree(str(tdir), eng)
            try:
                for k, (ranges, mode, mems) in enumerate([(ring_ranges(3), REF, [mem]), (ring_ranges(5), EXACT, [empty, mem]),
                                                          (ALL, REF, [mem, broken]), ([(5, 5), (0, 1 << 31)], EXACT, [])]):
                    out = tmp_path / f"out{k}"
                    want = tree.scan_ranges(ranges, mode, memtables=mems)
                    rows, stop = tree.scan_ranges_to_dir(ranges, str(out), mode, memtables=mems)
                    assert stop == want[3]
                    for r, row in enumerate(want[2]):
                        assert rows[r]["data_off"] == 0 and rows[r]["index_off"] == 0
                        assert {f: rows[r][f] for f in ("data_len", "index_len", "items")} == \
                               {f: row[f] for f in ("data_len", "index_len", "items")}
                        d = (out / f"{r}.data").read_bytes()
                        i = (out / f"{r}.index").read_bytes()
                        assert d == want[0][row["data_off"]:row["data_off"] + row["data_len"]].tobytes()
                        assert i == want[1][row["index_off"]:row["index_off"] + row["index_len"]].tobytes()
                    assert sorted(os.listdir(out)) == sorted(f"{r}.{x}" for r in range(len(ranges)) for x in ("data", "index"))
                    if mems and mems[-1] is broken:
                        assert stop == (len(tree.sstable_indices_and_sizes()) + 1, READ, 120)
                if eng is small:
                    assert small.stats()["partitions"] > 1
            finally:
                tree.close()
    finally:
        small.close()
