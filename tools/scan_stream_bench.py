#!/usr/bin/env python
"""Hash-range scans of a cfg2-shaped tree ON DISK: the whole-buffer path (LSMTree.scan_ranges: every file read whole into
pinned memory, uploaded whole, range-major outputs back in host memory) against the streamed path
(LSMTree.scan_ranges_to_dir: the files streamed through the engine's pinned rings partition by partition, every range
written to its own pair of files).  The tree: 8 SSTables of 1M entries of 305 bytes plus two 8192-entry memtable runs,
in a directory under /dev/shm (RAM-backed, so the file system is not what is measured).  Workloads as in
tools/scan_bench.py: (a) one EXACT arc, (b) the wrapped REFERENCE range, (c) three arcs.  Wall clock per call, --reps
calls, min / median / max; the partition count and ring size of the streamed path; byte parity of both paths against
the CPU scan oracle.  Also, for where the time goes: the whole-buffer path's H2D / kernel / D2H times (dbeel_last_stats)
and the time to read the tree's files once with one thread.
Usage: tools/scan_stream_bench.py [--reps 5] [--keys-per-run 1000000] [--out profiles/r04_scan_stream.json]"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import oracle  # noqa: E402
import scan_oracle  # noqa: E402  (parity only)
from bench import make_runs_parallel  # noqa: E402
from dbeel_b200 import capi, sstable  # noqa: E402
from dbeel_b200 import storage_engine as se  # noqa: E402
from dbeel_b200 import workloads as W  # noqa: E402
from tools.scan_bench import card  # noqa: E402


def read_dir_outputs(out_dir, n_ranges):
    d = b"".join(open(os.path.join(out_dir, f"{r}.data"), "rb").read() for r in range(n_ranges))
    i = b"".join(open(os.path.join(out_dir, f"{r}.index"), "rb").read() for r in range(n_ranges))
    return np.frombuffer(d, np.uint8), np.frombuffer(i, np.uint8)


def rebased(rows):
    """per_range rows of the streamed path (every range its own stream) as offsets into the concatenation."""
    out, d, i = [], 0, 0
    for r in rows:
        out.append(dict(r, data_off=d, index_off=i))
        d += r["data_len"]
        i += r["index_len"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--keys-per-run", type=int, default=1_000_000)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_scan_stream.json"))
    a = ap.parse_args()
    cfg = W.CFG2 if a.keys_per_run == 1_000_000 else W.scaled(W.CFG2, a.keys_per_run)
    work = tempfile.mkdtemp(prefix="dbeel_scan_stream_", dir=a.dir)
    try:
        t0 = time.time()
        runs = make_runs_parallel(cfg)
        mems = W.make_merge_runs(W.scaled(W.CFG2, 8192))[:2]  # flushing + active memtable as sorted runs
        tdir = os.path.join(work, "tree")
        os.makedirs(tdir)
        for k, run in enumerate(runs):  # SSTables 0, 2, 4, ... (lsm_tree.rs: flushes take even indices)
            sstable.write_run_files(tdir, 2 * k, run)
        files = [sstable.read_run_files(tdir, 2 * k) for k in range(len(runs))]
        tables = files + mems
        del runs
        print(f"tree written in {time.time() - t0:.1f} s: {len(tables)} tables, "
              f"{sum(d.size for d, _ in tables) / 1e9:.2f} GB .data under {tdir}", flush=True)
        t1 = time.time()
        for k in range(len(files)):
            sstable.read_run_files(tdir, 2 * k)
        read_once_s = time.time() - t1
        ring = sorted(oracle.murmur3_32(f"dbeel-{k}".encode()) for k in range(8))
        arcs = [(ring[k - 1], ring[k]) for k in range(1, 8)]
        arc_a = min(arcs, key=lambda r: abs((r[1] - r[0]) / 2**32 - 0.125))
        workloads = {
            "a_node_addition_1_exact_arc": ([arc_a], capi.SCAN_EXACT),
            "b_wrapped_reference_everything": ([(ring[7], ring[0])], capi.SCAN_REFERENCE),
            "c_three_ranges": (arcs[:3], capi.SCAN_EXACT),
        }
        eng = capi.Engine(0)
        tree = se.LSMTree(tdir, eng)
        name, plim = card()
        rec = {"workload": "scan_ranges of a cfg2-shaped tree on disk (/dev/shm): whole buffers vs streamed to files",
               "gpu": name, "power_limit": plim, "tables": len(tables),
               "entries_in": int(sum(i.size // 16 for _, i in tables)), "data_bytes_in": int(sum(d.size for d, _ in tables)),
               "reps": a.reps, "warmup": a.warmup, "stream_ring": int(os.environ.get("DBEEL_STREAM_RING", 3)),
               "partition_mb": int(os.environ.get("DBEEL_PARTITION_MB", 256)),
               "io_threads_env": os.environ.get("DBEEL_IO_THREADS"), "read_tree_files_once_one_thread_s": round(read_once_s, 3)}
        res = {}
        for wname, (ranges, mode) in workloads.items():
            exp = scan_oracle.scan_ranges(tables, ranges, mode)
            out_dir = os.path.join(work, "out")
            whole_s, stream_s, whole_st, stream_st = [], [], [], []
            for k in range(a.warmup + a.reps):
                t = time.time()
                got = tree.scan_ranges(ranges, mode, memtables=mems)
                dt = time.time() - t
                if k >= a.warmup:
                    whole_s.append(dt)
                    whole_st.append(eng.stats())
                shutil.rmtree(out_dir, ignore_errors=True)
                t = time.time()
                rows, stop = tree.scan_ranges_to_dir(ranges, out_dir, mode, memtables=mems)
                dt = time.time() - t
                if k >= a.warmup:
                    stream_s.append(dt)
                    stream_st.append(eng.stats())
            parity_whole = bool(np.array_equal(got[0], exp[0]) and np.array_equal(got[1], exp[1]) and got[2] == exp[2]
                                and got[3] == exp[3])
            sd, si = read_dir_outputs(out_dir, len(ranges))
            parity_stream = bool(np.array_equal(sd, exp[0]) and np.array_equal(si, exp[1]) and rebased(rows) == exp[2]
                                 and stop == exp[3])
            shutil.rmtree(out_dir, ignore_errors=True)
            ws = whole_st[int(np.argsort(whole_s)[len(whole_s) // 2])]
            ss = stream_st[int(np.argsort(stream_s)[len(stream_s) // 2])]
            res[wname] = {
                "ranges": [list(map(int, r)) for r in ranges], "mode": "EXACT" if mode else "REFERENCE",
                "entries_out": int(sum(r["items"] for r in rows)), "data_bytes_out": int(sum(r["data_len"] for r in rows)),
                "stop": list(stop),
                "whole_s": {"min": round(min(whole_s), 4), "median": round(float(np.median(whole_s)), 4), "max": round(max(whole_s), 4)},
                "stream_s": {"min": round(min(stream_s), 4), "median": round(float(np.median(stream_s)), 4), "max": round(max(stream_s), 4)},
                "speedup_median": round(float(np.median(whole_s) / np.median(stream_s)), 2),
                "whole_stage_ms_at_median": {k: round(ws[k], 3) for k in ("ms_h2d", "ms_total", "ms_d2h")},
                "stream_partitions": int(ss["partitions"]),
                "stream_stage_ms_at_median_summed_over_partitions": {k: round(ss[k], 3) for k in ("ms_h2d", "ms_total", "ms_d2h")},
                "parity_whole": parity_whole, "parity_stream": parity_stream,
            }
            print(wname, json.dumps(res[wname]), flush=True)
        rec["results"] = res
        rec["parity_all"] = all(r["parity_whole"] and r["parity_stream"] for r in res.values())
        tree.close()
        eng.close()
    finally:
        shutil.rmtree(work, ignore_errors=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"parity_all": rec["parity_all"], "out": a.out}))


if __name__ == "__main__":
    main()
