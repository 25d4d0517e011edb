#!/usr/bin/env python
"""Hash-range scans (dbeel_scan_ranges_device) over a cfg2-shaped tree resident in HBM: 8 SSTables of 1M entries of 305
bytes plus two 8192-entry memtable runs.  Three workloads:
  (a) node addition: one EXACT range = one arc of the dbeel-0..7 ring (~1/8 of the keys)
  (b) the wrapped REFERENCE range: every entry selected, the output-heavy bound
  (c) three ranges (step 2 of an addition): three arcs of the ring
Each: warm-up, then --reps timed calls (CUDA events on the engine stream), min / median / max, the per-stage split of
dbeel_last_stats, algorithmic bytes over the device-to-device copy peak measured in the same process, byte parity of the
last timed output against the CPU scan oracle; the oracle is timed on one core for (a).
Usage: tools/scan_bench.py [--reps 20] [--keys-per-run 1000000] [--out profiles/r03_scan_bench.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle  # noqa: E402
import scan_oracle  # noqa: E402  (parity + CPU baseline only)
from bench import hbm_peak, make_runs_parallel  # noqa: E402
from dbeel_b200 import capi  # noqa: E402
from dbeel_b200 import workloads as W  # noqa: E402


def card():
    try:  # read-only query
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim = [x.strip() for x in q.split(",")]
        return name, plim
    except Exception as ex:  # noqa: BLE001
        return f"unknown ({ex})", "unknown"


def copy_peak_gbs(dev, nbytes=2 << 30, reps=10):
    """Device-to-device copy, bytes read + written per second: the roofline the scan's bytes are divided by."""
    a = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * nbytes / (best * 1e-3) / 1e9


def header_bytes(runs):
    """Bytes classify reads per record: the 16-byte index record, the two length prefixes, the key, the timestamp."""
    total = 0
    for d, i in runs:
        idx = i.view("<u4").reshape(-1, 4)
        total += int((16 + 8 + 8 + 16 + (idx[:, 2].astype(np.int64) - 8)).sum())
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--keys-per-run", type=int, default=1_000_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_scan_bench.json"))
    a = ap.parse_args()
    cfg = W.CFG2 if a.keys_per_run == 1_000_000 else W.scaled(W.CFG2, a.keys_per_run)
    t0 = time.time()
    runs = make_runs_parallel(cfg)
    mems = W.make_merge_runs(W.scaled(W.CFG2, 8192))[:2]  # flushing + active memtable as sorted runs
    tables = list(runs) + mems
    print(f"tree built in {time.time() - t0:.1f} s: {len(tables)} tables, "
          f"{sum(d.size for d, _ in tables) / 1e9:.2f} GB .data", flush=True)
    dev = torch.device("cuda:0")
    peak = copy_peak_gbs(dev)
    t_tab = [(torch.from_numpy(d).to(dev), torch.from_numpy(i).to(dev)) for d, i in tables]
    ptrs = [(d.data_ptr(), d.numel(), i.data_ptr(), i.numel()) for d, i in t_tab]
    dc, ic = sum(d.size for d, _ in tables), 16 * sum(i.size // 16 for _, i in tables)
    od = torch.empty(dc + 32, dtype=torch.uint8, device=dev)
    oi = torch.empty(ic + 32, dtype=torch.uint8, device=dev)
    n_in = sum(i.size // 16 for _, i in tables)
    hdr = header_bytes(tables)
    ring = sorted(oracle.murmur3_32(f"dbeel-{k}".encode()) for k in range(8))
    arcs = [(ring[k - 1], ring[k]) for k in range(1, 8)]  # the seven arcs that do not wrap
    arc_a = min(arcs, key=lambda r: abs((r[1] - r[0]) / 2**32 - 0.125))
    workloads = {
        "a_node_addition_1_exact_arc": ([arc_a], capi.SCAN_EXACT),
        "b_wrapped_reference_everything": ([(ring[7], ring[0])], capi.SCAN_REFERENCE),
        "c_three_ranges": (arcs[:3], capi.SCAN_EXACT),
    }
    eng = capi.Engine(0)
    stream = torch.cuda.ExternalStream(eng.stream_ptr())
    rec = {"workload": "scan_ranges over a cfg2-shaped tree in HBM", "tables": len(tables), "entries_in": n_in,
           "data_bytes_in": int(dc), "reps": a.reps, "warmup": a.warmup}
    name, plim = card()
    rec["gpu"] = name
    rec["power_limit"] = plim
    rec["copy_peak_gbs_measured"] = round(peak, 1)
    rec["hbm_peak_gbs_bench"] = hbm_peak()[0]
    res = {}
    for wname, (ranges, mode) in workloads.items():
        call = lambda: eng.scan_ranges_device(ptrs, ranges, (od.data_ptr(), dc, oi.data_ptr(), ic), mode)  # noqa: E731
        for _ in range(a.warmup):
            call()
        ms, stages = [], []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            dl, il, rows, stop = call()
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
            stages.append(eng.stats())
        n_out = sum(r["items"] for r in rows)
        alg = hdr + 2 * dl + 16 * n_out
        med = float(np.median(ms))
        st = stages[int(np.argsort(ms)[len(ms) // 2])]
        gd, gi = od[:dl].cpu().numpy(), oi[:il].cpu().numpy()
        t1 = time.time()
        ed, ei, erows, estop = scan_oracle.scan_ranges(tables, ranges, mode)
        t_orc = time.time() - t1
        parity = bool(np.array_equal(gd, ed) and np.array_equal(gi, ei) and rows == erows and stop == estop)
        res[wname] = {
            "ranges": [list(map(int, r)) for r in ranges], "mode": "EXACT" if mode else "REFERENCE",
            "entries_out": n_out, "selected_frac": round(n_out / n_in, 4), "data_bytes_out": int(dl), "stop": list(stop),
            "ms_min": round(min(ms), 4), "ms_median": round(med, 4), "ms_max": round(max(ms), 4),
            "stage_ms_at_median": {k: round(st[k], 4) for k in ("ms_extract", "ms_resolve", "ms_gather", "ms_total")},
            "classify_ns_per_entry": round(st["ms_extract"] * 1e6 / n_in, 4),
            "algorithmic_bytes": int(alg), "algorithmic_gbs_at_median": round(alg / (med * 1e-3) / 1e9, 1),
            "frac_of_copy_peak": round(alg / (med * 1e-3) / 1e9 / peak, 3),
            "oracle_s_one_core": round(t_orc, 3), "parity": parity,
        }
        print(wname, json.dumps(res[wname]), flush=True)
    rec["results"] = res
    rec["parity_all"] = all(r["parity"] for r in res.values())
    eng.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"parity_all": rec["parity_all"], "out": a.out}))


if __name__ == "__main__":
    main()
