"""The partition plan of the streamed hash-range scan (dbeel_b200/csrc/host/scan_plan.h, built by g++ through
tests/scan_plan_shim.cc) against a Python restatement of its rules, on the random and damaged trees of
test_scan_ranges.py.  CPU only."""
import ctypes as C
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

from test_scan_ranges import DAMAGES, READ, damage, py_scan, random_tree

HERE = os.path.dirname(os.path.abspath(__file__))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("plan") / "scan_plan_shim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "scan_plan_shim.cc")])
    L = C.CDLL(so)
    L.shim_scan_plan.restype = C.c_int
    L.shim_scan_plan.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                 C.c_uint64, C.c_void_p]
    return L


def plan(shim, tables, budget):
    keep = [(np.ascontiguousarray(d, np.uint8), np.ascontiguousarray(i, np.uint8)) for d, i in tables]
    n_rec = sum(i.size // 16 for _, i in keep)
    dl = np.array([d.size for d, _ in keep] or [0], np.uint64)
    n = np.array([i.size // 16 for _, i in keep] or [0], np.uint64)
    ptrs = (C.c_void_p * max(1, len(keep)))(*[i.ctypes.data for _, i in keep])
    cap = n_rec + len(keep) + 1
    pieces, parts, summary = np.zeros(6 * cap, np.uint64), np.zeros(4 * cap, np.uint64), np.zeros(6, np.uint64)
    assert shim.shim_scan_plan(len(keep), dl.ctypes.data, ptrs, n.ctypes.data, budget, pieces.ctypes.data, cap,
                               parts.ctypes.data, cap, summary.ctypes.data) == 0
    n_pieces, n_parts = int(summary[0]), int(summary[1])
    stop = (int(summary[4]), READ, int(summary[5])) if summary[3] else None
    return ([tuple(int(v) for v in pieces[6 * k:6 * k + 6]) for k in range(n_pieces)],
            [tuple(int(v) for v in parts[4 * c:4 * c + 4]) for c in range(n_parts)], int(summary[2]), stop)


def records(tables):
    """(table, record, offset, full_size) in iteration order."""
    for t, (_, i) in enumerate(tables):
        b = bytes(i)
        for r in range(len(b) // 16):
            off, _ks, fs = struct.unpack_from("<QII", b, 16 * r)
            yield t, r, off, fs


def read_stop(tables):
    """The first record (or table without one) the reference cannot read: (table, READ, record), or None."""
    for t, (d, i) in enumerate(tables):
        if i.size // 16 == 0:
            return (t, READ, 0)
        for _, r, off, fs in (x for x in records([(d, i)])):
            if fs == 0 or off + fs > d.size:
                return (t, READ, r)
    return None


def check_plan(tables, budget, pieces, parts, scheduled, stop):
    """The planner's rules (scan_plan.h), restated."""
    assert stop == read_stop(tables)
    recs = list(records(tables))
    if stop is not None:
        t0, _, r0 = stop
        recs = [x for x in recs if (x[0], x[1]) < (t0, r0)]
    assert scheduled == len(recs)
    # every record before the stop lies in exactly one partition, in iteration order
    walked = []
    for part, t, lo, hi, slo, shi in pieces:
        walked += [(part, t, r) for r in range(lo, hi)]
    assert [(t, r) for _, t, r in walked] == [(t, r) for t, r, _, _ in recs]
    assert [p for p, _, _ in walked] == sorted(p for p, _, _ in walked)
    by_rec = {(t, r): (off, fs) for t, r, off, fs in recs}
    ordinal = 0
    for c, (first, n, span_bytes, data_bytes) in enumerate(parts):
        mine = [pc for pc in pieces if pc[0] == c]
        assert first == ordinal and n == sum(hi - lo for _, _, lo, hi, _, _ in mine) and n > 0
        assert len({t for _, t, _, _, _, _ in mine}) == len(mine)  # one piece per table
        ordinal += n
        assert span_bytes == sum(shi - slo for *_, slo, shi in mine)
        assert data_bytes == sum(by_rec[(t, r)][1] for _, t, lo, hi, _, _ in mine for r in range(lo, hi))
        for _, t, lo, hi, slo, shi in mine:  # every record's bytes inside its piece's span, and the span is tight
            offs = [by_rec[(t, r)] for r in range(lo, hi)]
            assert all(slo <= off and off + fs <= shi for off, fs in offs)
            assert slo == min(off for off, _ in offs) and shi == max(off + fs for off, fs in offs)
        assert 16 * n + span_bytes <= budget or n == 1, (c, n, span_bytes, budget)
    assert ordinal == scheduled


@pytest.mark.parametrize("seed", range(8))
def test_plan_random_trees(shim, seed):
    rng = np.random.default_rng(300 + seed)
    tables = random_tree(rng, int(rng.integers(1, 7)), 60, n_mem=int(rng.integers(0, 3)))
    total = sum(d.size + i.size for d, i in tables)
    for budget in (1, 64, 300, 4096, total // 3 + 1, total + 1, 1 << 40):
        pieces, parts, scheduled, stop = plan(shim, tables, budget)
        check_plan(tables, budget, pieces, parts, scheduled, stop)
        if budget >= total:
            assert len(parts) == 1
        if budget == 1:
            assert len(parts) == scheduled  # every record alone
    pieces, parts, scheduled, stop = plan(shim, tables, 4096)
    assert any(len({t for p, t, *_ in pieces if p == c}) > 1 for c in range(len(parts))) or len(tables) == 1


@pytest.mark.parametrize("kind", DAMAGES)
def test_plan_stops_like_the_restatement(shim, kind):
    rng = np.random.default_rng(400 + DAMAGES.index(kind))
    for trial in range(6):
        tables = damage(rng, random_tree(rng, 4, 50), kind)
        for budget in (200, 2048, 1 << 30):
            pieces, parts, scheduled, stop = plan(shim, tables, budget)
            check_plan(tables, budget, pieces, parts, scheduled, stop)
            _, want = py_scan(tables, [])
            if kind in ("zero", "eof", "empty"):
                assert stop == want
            else:  # a DECODE stop is the device's to find: the planner schedules through it
                assert stop is None


def test_plan_scattered_offsets_split_partitions(shim):
    rng = np.random.default_rng(9)
    tables = random_tree(rng, 3, 200, n_mem=0)
    budget = sum(d.size + i.size for d, i in tables) // 4
    _, parts, _, _ = plan(shim, tables, budget)
    scattered = []
    for d, i in tables:  # the same records, listed in a permuted order: still readable, no longer adjacent
        rec = i.reshape(-1, 16)
        scattered.append((d, rec[rng.permutation(len(rec))].reshape(-1).copy()))
    pieces, sparts, scheduled, stop = plan(shim, scattered, budget)
    check_plan(scattered, budget, pieces, sparts, scheduled, stop)
    assert stop is None and len(sparts) > len(parts)


def test_plan_empty_inputs(shim):
    assert plan(shim, [], 4096) == ([], [], 0, None)
    empty = (np.zeros(0, np.uint8), np.zeros(0, np.uint8))
    assert plan(shim, [empty], 4096) == ([], [], 0, (0, READ, 0))
