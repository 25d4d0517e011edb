"""bench.py --workload cfg5 (BASELINE.json configs[4]) and its checker: the product pipeline is dbeel_b200/cfg5.py; this
file adds what only tests and benches may touch -- the CPU oracle replay of every shard and the byte comparison."""
from __future__ import annotations

import json
import time

import numpy as np

from dbeel_b200 import capi
from dbeel_b200 import storage_engine as se
from dbeel_b200.cfg5 import (CAPACITY, CFG5_IDS, CFG5_WRITES, DOC_BYTES, FACTOR, N_SHARDS, ZIPF_S, build_stream_device, own_positions, ring_arcs,
                             pipeline, stream_ids)

# ------------------------------------------------------------------------------------ the checker

def check_against_oracle(res, data_host: np.ndarray, routed_host: np.ndarray, capacity: int = CAPACITY, threads: int = 8):
    """Replays every own shard on the CPU oracle (red-black-tree memtables, the recorded plan) and compares every table left,
    byte for byte.  Returns (all identical, cpu seconds of the slowest shard thread, total cpu seconds)."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor

    def one(pos):
        t = time.perf_counter()
        lo = int(res["starts"][pos])
        cnt = int(res["starts"][pos + 1]) - lo
        dense = oracle.densify(data_host, routed_host[16 * lo:16 * (lo + cnt)])
        flushed = oracle.memtable_flushes(dense, capacity=capacity, emulate_page_cache=True)
        if [c for _, c in res["mem"][pos]] != _arrivals_per_flush(dense, flushed, capacity, oracle):
            return False, time.perf_counter() - t, "memtable boundaries differ"
        otab = {2 * m: (d, i, n, None) for m, (d, i, n) in enumerate(flushed)}
        for indices, out_index, keep, seed in res["plan"][pos]:
            d, i, b, n = oracle.compact([(otab[k][0], otab[k][1]) for k in indices], keep, seed=seed, emulate_page_cache=True)
            for k in indices:
                del otab[k]
            otab[out_index] = (d, i, n, b)
        cpu_s = time.perf_counter() - t
        gt = res["tables"][pos]
        if sorted(gt) != sorted(otab):
            return False, cpu_s, "table sets differ"
        for k in sorted(gt):
            g, o = gt[k], otab[k]
            if g[2] != o[2] or not np.array_equal(g[0].cpu().numpy(), o[0]) or not np.array_equal(g[1].cpu().numpy(), o[1]):
                return False, cpu_s, f"table {k} differs"
            if (g[3] is None) != (o[3] is None) or (g[3] is not None and not np.array_equal(g[3].cpu().numpy(), o[3])):
                return False, cpu_s, f"bloom of table {k} differs"
        return True, cpu_s, ""

    with ThreadPoolExecutor(max_workers=max(1, min(threads, len(res["mem"])))) as ex:
        outs = list(ex.map(one, list(res["mem"])))
    why = [w for ok, _, w in outs if not ok]
    return all(ok for ok, _, _ in outs), max(s for _, s, _ in outs), sum(s for _, s, _ in outs), why


def _arrivals_per_flush(dense, flushed, capacity, oracle):
    """Arrivals each of the oracle's memtables absorbed (the tree fills at `capacity` distinct keys)."""
    out, pos, n = [], 0, dense[1].size // 16
    while pos < n:
        m = se.memtable_cut(dense, pos, capacity)
        out.append(m)
        pos += m
    assert len(out) == len(flushed)
    return out


# ------------------------------------------------------------------------------------ bench entry points

def run_one_shard(eng, torch, dev, n_writes: int = 1_500_000):
    """other_configs evidence in the default bench line: a scaled cfg5 stream through the full pipeline on one GPU."""
    ids, tomb = stream_ids(n_writes, max(8192, n_writes // 4))
    data, index, total = build_stream_device(torch, dev, ids, tomb)
    ring, _ = capi.shard_ring(N_SHARDS)
    pipeline(eng, torch, dev, data, index, ring, own_positions(0, 1))  # warm-up (allocator, workspaces)
    res = pipeline(eng, torch, dev, data, index, ring, own_positions(0, 1))
    ok, cpu_max, cpu_sum, why = check_against_oracle(res, data.cpu().numpy(), res["routed"][:index.numel()].cpu().numpy())
    nbytes = total + index.numel()
    return {"workload": f"cfg5 scaled: {n_writes} Zipf(0.99) writes x {DOC_BYTES} B docs -> {N_SHARDS} shards by murmur3 ring, 1 GPU",
            "arrival_bytes": nbytes, "memtables": res["memtables"], "compactions": res["compactions"], "picker_rounds": res["rounds"],
            "kernel_ms": round(res["kernel_ms"], 3), "wall_ms": round(res["wall_ms"], 3), "stage_ms": {k: round(v, 3) for k, v in res["ms"].items()}, "flush_calls": res["flush_calls"], "flush_stage_ms": res["flush_stage_ms"],
            "value": round(nbytes / 1e6 / (res["wall_ms"] / 1e3), 1), "unit": "MB/s of arrivals (wall clock, picker and allocations included)",
            "kernel_value": round(nbytes / 1e6 / (res["kernel_ms"] / 1e3), 1),
            "cpu_oracle_mbs": round(nbytes / 1e6 / cpu_sum, 1), "cpu_threads": 1, "short_memtables": len(res["short"]),
            "parity_vs_oracle": bool(ok and not res["short"]), "why": why}


def bench(args, torch, dist, dev, rank, world, local, ClockSampler, hbm_peak, METRIC, UNIT, log):
    """`bench.py --workload cfg5`: the full configs[4] stream on N GPUs; one JSON line from rank 0."""
    n_writes = args.writes or CFG5_WRITES
    n_ids = CFG5_IDS if n_writes >= CFG5_WRITES else max(8192, n_writes // 4)
    t = time.time()
    ids, tomb = stream_ids(n_writes, n_ids)
    data, index, total = build_stream_device(torch, dev, ids, tomb)
    torch.cuda.synchronize()
    log(f"[cfg5 r{rank}] {n_writes} arrivals, {total / 1e9:.2f} GB of .data resident in HBM ({time.time() - t:.0f}s)")
    eng = capi.Engine(local)
    ring, ring_ids = capi.shard_ring(N_SHARDS)
    mine = own_positions(rank, world, ring)
    steps = args.steps
    warm = max(1, min(args.warmup, 2))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warm):
        res = pipeline(eng, torch, dev, data, index, ring, mine)
        del res
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    kernel_ms = 0.0
    launches = 0
    for _ in range(steps):
        res = pipeline(eng, torch, dev, data, index, ring, mine)
        kernel_ms += res["kernel_ms"]
        launches += res["launches"]
        if _ + 1 < steps:
            del res
    barrier()
    t1 = time.perf_counter()
    sampler.stop()
    clocks = sampler.summary(t0, t1)
    wall_ms = (t1 - t0) * 1e3
    own_bytes = res["own_arrival_bytes"]
    tm = torch.tensor([wall_ms, kernel_ms], dtype=torch.float64, device=dev)
    sm = torch.tensor([float(own_bytes), float(launches), float(res["memtables"]), float(res["compactions"]), float(len(res["short"]))],
                      dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    # parity of every rank's shards (outside the timed region)
    parity, cpu_max, cpu_sum = None, 0.0, 0.0
    if not args.no_cpu:
        ok, cpu_max, cpu_sum, why = check_against_oracle(res, data.cpu().numpy(), res["routed"][:index.numel()].cpu().numpy())
        parity = bool(ok and not res["short"])
        log(f"[cfg5 r{rank}] parity of {len(mine)} shard(s) vs the oracle: {parity} {why} (cpu {cpu_sum:.1f}s)")
    par = torch.tensor([1.0 if parity in (True, None) else 0.0, cpu_max, cpu_sum], dtype=torch.float64, device=dev)
    if world > 1:
        pm = par.clone()
        dist.all_reduce(par, op=dist.ReduceOp.MIN)
        dist.all_reduce(pm, op=dist.ReduceOp.MAX)
        cs = torch.tensor([cpu_sum], dtype=torch.float64, device=dev)
        dist.all_reduce(cs, op=dist.ReduceOp.SUM)
        cpu_max, cpu_sum = float(pm[1]), float(cs[0])
    if rank == 0:
        total_bytes = float(sm[0])
        value = total_bytes * steps / 1e6 / (float(tm[0]) / 1e3)
        line = {"metric": "cfg5 pipeline throughput MB/s (arrival bytes: .data + .index of the write stream)", "value": round(value, 1),
                "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": round(float(tm[0]) / steps, 3),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": f"cfg5: {n_writes} Zipf({ZIPF_S}) writes over {n_ids} keys x {DOC_BYTES} B docs, {N_SHARDS} shards by "
                                       f"murmur3_32 ring of dbeel-0..7, memtables of {CAPACITY} keys, size-tiered picker factor {FACTOR}",
                           "arrival_bytes": int(total_bytes), "memtables": int(sm[2]), "compactions": int(sm[3]),
                           "ring_positions_rank0": [int(x) for x in mine], "ring_ids": [int(x) for x in ring_ids],
                           "ring_arcs": [round(float(x), 4) for x in ring_arcs(ring)],
                           "placement": "ring positions dealt out by arc length, longest first, each to the least loaded rank",
                           "timing": "wall clock of route + cut + flush waves + picker rounds per rank (device synchronised), max over ranks"},
                "kernel_ms_per_step": round(float(tm[1]) / steps, 3),
                "kernel_value": round(total_bytes * steps / 1e6 / (float(tm[1]) / 1e3), 1),
                "stage_ms_rank0": {k: round(v, 3) for k, v in res["ms"].items()},
                "gpu_launches": int(sm[1]), "clocks": clocks,
                "cpu_baseline": None if parity is None else {"value": round(total_bytes / 1e6 / cpu_max, 1), "unit": UNIT, "cores": N_SHARDS, "kind": "port",
                                                             "sample": f"the same stream: one oracle thread per shard (red-black-tree memtables + the recorded "
                                                                       f"compaction plan), slowest shard {cpu_max:.1f} s, all shards {cpu_sum:.1f} cpu-s"},
                "short_memtables": int(sm[4]),
                "parity_vs_oracle": None if parity is None else bool(par[0] > 0.5), "parity_all_ranks": None if parity is None else bool(par[0] > 0.5)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
