#!/usr/bin/env python
"""bench.py -- compaction throughput (MB/s of input bytes) of the B200 engine vs the CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic input: the 8 independent shard
compactions of BASELINE.json configs[3] -- each one configs[1]'s 8-way merge of 1M-key x 256-byte-doc
runs ("cfg2" shape: 2.55 GB of .data+.index in, bloom on, tombstones dropped; seeds 40..47).  The 8 jobs
are the same at every N: rank r runs the jobs of shards r, r+N, ... one after the other (8 / 4 / 2 / 1
jobs per GPU at N = 1 / 2 / 4 / 8, SURVEY.md section 8e), so N = 1 does the same work as N = 8 (strong
scaling, no data-path collective; NCCL only hands the job table out, closes the barriers and reduces the
report).  Per-job figures (ms_per_job, stage_ms, roofline) are configs[1]'s.

`value`    whole-job MB/s of input bytes with the runs resident in HBM (all kernels of the
           pipeline; timed with CUDA events on the engine's stream, max over ranks)
`e2e`      the same metric through dbeel_compact() with HOST (pinned) buffers: H2D of the runs
           and D2H of the output SSTable inside the timed region
`roofline` the dominant kernel (k_gather): algorithmic bytes / its CUDA-event time vs the
           measured HBM copy peak
`cpu_baseline` the CPU oracle (port of the reference's single-threaded compact()) on one core

--impl reference times the CPU path alone with every host core busy (one full-size shard compaction
per core, the way dbeel's thread-per-core runtime would run them).
--workload cfg5 runs BASELINE.json configs[4] instead (dbeel_b200/cfg5.py).
--dump-outputs DIR writes what the jobs of the last timed step returned (either arm; see dump_job_outputs).  The inputs
are seeded, so two builds run with the same arguments can be compared file for file.  The GPU arm then gives every job
its own output buffers (8 x ~2.5 GB more HBM), so its timed kernels write elsewhere than in a run without the flag; the
JSON line says so under "dump_outputs".  The reference arm dumps the jobs its last step ran, all 8 only when it ran 8.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "compaction throughput MB/s (input bytes) at 1/2/4/8 B200 vs CPU shards"
UNIT = "MB/s"
SEED32 = bytes(range(32))
FALLBACK_HBM_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
GATHER_KERNEL = "k_gather"
SEED32_DEFAULT_MIN = 1_048_576  # oracle.compact's bloom_min_size positional (mod.rs:19)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def gather_traffic_from_profile():
    """(dram read+write bytes per gather launch, the ncu capture it was read from) from the committed summary, if any."""
    p = os.path.join(ROOT, "profiles", "gather_traffic.json")
    try:
        with open(p) as f:
            j = json.load(f)
        return j.get("dram_bytes_per_launch"), j.get("source")
    except Exception:
        return None, None


# ------------------------------------------------------------------------------------ clocks

class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, device_index: int, period_s: float = 0.01):
        self.samples = []
        self.marks = []
        self._stop = threading.Event()
        self._period = period_s
        self._ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = device_index
            if vis:
                try:
                    phys = int(vis.split(",")[device_index])
                except Exception:
                    phys = device_index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
            self._ok = True
        except Exception as ex:  # pragma: no cover
            log(f"[bench] NVML unavailable ({ex}); clocks not sampled")
            self.max_mhz = None
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:
                pass
            time.sleep(self._period)

    def start(self):
        if self._ok:
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._ok:
            self._t.join(timeout=2)

    def summary(self, t0: float, t1: float) -> dict:
        if not self._ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        if not inside:  # region shorter than the sampling period: take the nearest samples
            inside = sorted(self.samples, key=lambda s: min(abs(s[0] - t0), abs(s[0] - t1)))[:3]
        mhz = sorted(s[1] for s in inside)
        bits = 0
        for s in inside:
            bits |= s[2]
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if bits & b), "samples": len(inside)}


# ------------------------------------------------------------------------------------ workload

N_JOBS = 8  # BASELINE.json configs[3]: 8 independent shard compactions, the same 8 at every N
WORKLOAD_NAME = "cfg4: 8 independent shard compactions, each cfg2-shaped (8-way, 1M keys/run, 256 B docs; seeds 40-47)"


def common_config():
    """The part of `config` both arms print (the driver compares the two)."""
    return {"workload": WORKLOAD_NAME, "runs": 8, "keys_per_run": 1_000_000, "doc_bytes": 256, "jobs": N_JOBS,
            "keep_tombstones": False, "bloom": True}


def job_config(job, workload: str = "cfg2"):
    from dbeel_b200 import workloads as W
    if workload == "cfg3":  # BASELINE.json configs[2]: not the headline, kept for cross-checks
        return W.CFG3
    return W.cfg4_shard(job.shard_id)


def make_runs_parallel(cfg):
    """make_merge_runs, one thread per run (numpy releases the GIL in the heavy parts)."""
    from concurrent.futures import ThreadPoolExecutor

    from dbeel_b200 import workloads as W

    def one(r):
        rng = np.random.default_rng([cfg.seed, r])
        ids = W._run_ids(cfg, rng, r)
        keys = W.format_keys(ids)
        dense = W._dense_rows([cfg.seed, r, 7], ids.shape[0], keys.shape[1], cfg.doc_bytes)
        tomb = rng.random(ids.shape[0]) < cfg.tombstone_frac
        ts = W.BASE_TS + (np.int64(r) * ids.shape[0] + rng.permutation(ids.shape[0]).astype(np.int64)) * 1000
        from dbeel_b200.sstable import build_run_dense
        return build_run_dense(dense, keys, ts, tomb)

    with ThreadPoolExecutor(max_workers=min(cfg.n_runs, os.cpu_count() or 1)) as ex:
        return list(ex.map(one, range(cfg.n_runs)))


def same_output(a, b) -> bool:
    """(data, index, bloom | None, items) of the engine vs the oracle, byte for byte."""
    return bool(a[3] == b[3] and np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
                and (a[2] is None) == (b[2] is None) and (a[2] is None or np.array_equal(a[2], b[2])))


DUMP_SAMPLE = {"data": 1 << 20, "index": 1 << 18, "bloom": 1 << 18}  # bytes of each output file sampled per job
DUMP_BLOCK = 1 << 16  # bytes per block sum


def dump_job_outputs(out_dir: str, shard_id: int, data, index, bloom, items: int) -> None:
    """--dump-outputs: one job's output SSTable (uint8 torch tensors on any device, bloom None when there is none) as .npy
    files that two builds can be compared with, file for file:
      job<i>_lengths.npy          float64 [.data bytes, .index bytes, .bloom bytes, entries written]
      job<i>_<file>_sample.npy    float32 bytes of the file at positions drawn from a fixed seed (the whole file if smaller)
      job<i>_<file>_blocksum.npy  float64 sum of the bytes of every 64 KiB block (exact: a changed byte moves one of them)
    About 6.6 MB per job of the default workload, 53 MB for its 8 jobs."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    files = {"data": data, "index": index, "bloom": bloom if bloom is not None else torch.zeros(0, dtype=torch.uint8)}
    np.save(os.path.join(out_dir, f"job{shard_id}_lengths.npy"), np.array([t.numel() for t in files.values()] + [items], np.float64))
    for k, (name, t) in enumerate(files.items()):
        n = t.numel()
        if n <= DUMP_SAMPLE[name]:
            sample = t
        else:
            pos = np.sort(np.random.default_rng([shard_id, k]).integers(0, n, DUMP_SAMPLE[name]))
            sample = t[torch.from_numpy(pos).to(t.device)]
        whole = n - n % DUMP_BLOCK
        sums = t[:whole].view(-1, DUMP_BLOCK).sum(1, dtype=torch.float64)
        if n > whole:
            sums = torch.cat([sums, t[whole:].sum(dtype=torch.float64).view(1)])
        np.save(os.path.join(out_dir, f"job{shard_id}_{name}_sample.npy"), sample.cpu().numpy().astype(np.float32))
        np.save(os.path.join(out_dir, f"job{shard_id}_{name}_blocksum.npy"), sums.cpu().numpy())


# ------------------------------------------------------------------------------------ GPU arm

def device_resident_job(eng, torch, dev, runs, opts, steps, warmup):
    """One compaction, inputs and outputs in HBM: (sum of CUDA-event ms over `steps`, stage sums, last stats, result)."""
    from dbeel_b200 import capi
    dc, ic, bc = capi.compact_bound([(d.size, i.size) for d, i in runs], opts)
    t_runs = [(torch.from_numpy(d).to(dev), torch.from_numpy(i).to(dev)) for d, i in runs]
    od = torch.empty(dc + 16, dtype=torch.uint8, device=dev)
    oi = torch.empty(ic + 16, dtype=torch.uint8, device=dev)
    ob = torch.empty(bc + 16, dtype=torch.uint8, device=dev)
    d_runs = [(d.data_ptr(), d.numel(), i.data_ptr(), i.numel()) for d, i in t_runs]
    d_out = (od.data_ptr(), dc, oi.data_ptr(), ic, ob.data_ptr(), bc)
    for _ in range(warmup):
        res = eng.compact_device(d_runs, d_out, opts)
    ms = 0.0
    stage = {"ms_extract": 0.0, "ms_merge": 0.0, "ms_resolve": 0.0, "ms_gather": 0.0}
    for _ in range(steps):
        res = eng.compact_device(d_runs, d_out, opts)
        st = eng.stats()
        ms += st["ms_total"]
        for k in stage:
            stage[k] += st[k]
    out = (od[:res[0]].cpu().numpy(), oi[:res[1]].cpu().numpy(), ob[:res[2]].cpu().numpy() if res[2] else None, res[3])
    return ms, stage, eng.stats(), out


def file_fed_job(eng, expected):
    """Row N3, the storage edge: one headline job (shard 0 of configs[3]) file to file through dbeel_tree_compact on tmpfs --
    open, read, H2D, kernels, D2H, write, journal, renames, all inside the timed call.  Streamed through the engine's pinned
    rings (dbeel_compact_stream, the default) against the same call reading every file whole first (DBEEL_TREE_STREAM=0)."""
    import shutil
    import tempfile
    from dbeel_b200 import sstable, storage_engine as se
    from dbeel_b200 import workloads as W
    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    if shutil.disk_usage(base).free < 12e9:
        return {"skipped": f"less than 12 GB free under {base}"}
    cfg = W.cfg4_shard(0)
    runs = make_runs_parallel(cfg)
    in_bytes = sstable.input_bytes(runs)
    root = tempfile.mkdtemp(prefix="dbeel_file_fed_", dir=base)
    try:
        master = os.path.join(root, "master")
        os.makedirs(master)
        for r, run in enumerate(runs):
            sstable.write_run_files(master, 2 * r, run)
        del runs
        idx = [2 * r for r in range(cfg.n_runs)]
        out_index = 2 * cfg.n_runs - 1

        def one(tag, streamed):
            d = os.path.join(root, tag)
            os.makedirs(d)
            for name in os.listdir(master):  # hard links: the tree deletes its inputs, the bytes stay in `master`
                os.link(os.path.join(master, name), os.path.join(d, name))
            os.environ["DBEEL_TREE_STREAM"] = "1" if streamed else "0"
            tree = se.LSMTree(d, eng)
            t0 = time.perf_counter()
            tree.compact(idx, out_index, cfg.keep_tombstones, bloom_seed=SEED32)
            dt = time.perf_counter() - t0
            st = eng.stats()
            tree.close()
            return d, dt, st

        res = {"workload": cfg.name + ", files on tmpfs (" + base + ")", "input_bytes": in_bytes, "unit": UNIT}
        _, _, _ = one("warm", True)  # the rings are page-locked on first use (grow-only)
        shutil.rmtree(os.path.join(root, "warm"))
        best = None
        for k in range(3):
            d, dt, st = one(f"s{k}", True)
            best = dt if best is None else min(best, dt)
            if k < 2:
                shutil.rmtree(d)
        res["streamed"] = {"value": round(in_bytes / 1e6 / best, 1), "ms": round(best * 1e3, 1), "partitions": st["partitions"],
                           "api": "dbeel_tree_compact -> dbeel_compact_stream (pread threads -> pinned ring -> H2D / kernels / D2H -> pinned ring -> writer threads copying into the mapped output files)"}
        if expected is not None:
            gd, gi = sstable.read_run_files(d, out_index)
            gb = np.fromfile(os.path.join(d, sstable.file_name(out_index, "bloom")), dtype=np.uint8)
            res["parity_vs_oracle"] = bool(np.array_equal(gd, expected[0]) and np.array_equal(gi, expected[1]) and
                                           expected[2] is not None and np.array_equal(gb, expected[2]))
            del gd, gi, gb
        shutil.rmtree(d)
        d, dt, st = one("whole", False)
        res["whole_buffers"] = {"value": round(in_bytes / 1e6 / dt, 1), "ms": round(dt * 1e3, 1),
                                "api": "dbeel_tree_compact, DBEEL_TREE_STREAM=0: files read whole into fresh pinned buffers, dbeel_compact, files written"}
        return res
    finally:
        os.environ.pop("DBEEL_TREE_STREAM", None)
        shutil.rmtree(root, ignore_errors=True)


def other_configs(eng, torch, dev, peak):
    """Evidence for the configs that are not the headline, outside every timed headline region (rank 0, N = 1)."""
    import oracle
    from dbeel_b200 import capi, sstable
    from dbeel_b200 import workloads as W
    out = {}
    # configs[0]: the reference's own CPU-runnable case, host entry point
    runs = W.make_merge_runs(W.CFG1)
    got = eng.compact(runs, False, seed=SEED32)
    out["cfg1"] = {"workload": W.CFG1.name, "parity_vs_oracle": same_output(got, oracle.compact(runs, False, seed=SEED32)),
                   "entries_out": got[3]}
    # configs[2]: full size, device-resident
    t = time.time()
    runs = make_runs_parallel(W.CFG3)
    opts = capi.make_opts(W.CFG3.keep_tombstones, seed=SEED32)
    steps = 10
    ms, stage, st, got = device_resident_job(eng, torch, dev, runs, opts, steps, 3)
    algo = st["input_bytes"] + st["output_bytes"]
    exp = oracle.compact(runs, W.CFG3.keep_tombstones, seed=SEED32, emulate_page_cache=True)
    out["cfg3"] = {"workload": W.CFG3.name, "input_bytes": st["input_bytes"], "ms_per_step": round(ms / steps, 4),
                   "value": round(st["input_bytes"] / 1e6 / (ms / steps / 1e3), 1), "unit": UNIT,
                   "stage_ms": {k: round(v / steps, 4) for k, v in stage.items()},
                   "pipeline_roofline": {"algo_bytes": algo, "frac": round(algo / 1e9 / (ms / steps / 1e3) / peak, 4),
                                         "read_only_frac": round(st["input_bytes"] / 1e9 / (ms / steps / 1e3) / peak, 4)},
                   "parity_vs_oracle": same_output(got, exp), "entries_out": got[3]}
    log(f"[bench] other configs: cfg1 parity {out['cfg1']['parity_vs_oracle']}, cfg3 {out['cfg3']['ms_per_step']} ms/step "
        f"parity {out['cfg3']['parity_vs_oracle']} ({time.time() - t:.0f}s)")
    del runs, got, exp
    try:  # row N3: the headline job file to file -- in a child process with a deadline, so that nothing on that path (threads,
        # files, a full tmpfs) can take the headline line down with it
        import subprocess
        t = time.time()
        cp = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "file_fed.py"), "--parity"], capture_output=True, text=True, timeout=240)
        lines = [ln for ln in cp.stdout.splitlines() if ln.startswith("{")]
        out["file_fed"] = json.loads(lines[-1]) if cp.returncode == 0 and lines else {"error": f"rc {cp.returncode}: {cp.stderr[-300:]}"}
        log(f"[bench] file-fed job: {out['file_fed']} ({time.time() - t:.0f}s)")
    except Exception as ex:  # pragma: no cover
        out["file_fed"] = {"error": repr(ex)}
    try:  # configs[4], one shard's stream (the 8-GPU run is --workload cfg5)
        import bench_cfg5
        out["cfg5_scaled"] = bench_cfg5.run_one_shard(eng, torch, dev, n_writes=1_500_000)
    except Exception as ex:  # pragma: no cover
        out["cfg5_scaled"] = {"error": repr(ex)}
    return out


def spread_device(local_rank: int, local_world: int) -> int:
    """Which GPU of the node a rank drives.  With fewer ranks than GPUs the ranks are spread evenly over the node (rank r ->
    GPU r * n_gpus / N: 0,4 for two ranks, 0,2,4,6 for four) instead of packed onto GPUs 0..N-1: host-memory DMA is capped per
    CPU socket (profiles/r02_pcie_topology.txt: 91 GB/s for one GPU, 155 for two and 189 for four on ONE socket, 379 for all
    eight over both), so ranks that share a socket share that cap and the end-to-end path is the first to feel it."""
    try:
        import pynvml
        pynvml.nvmlInit()
        n_dev = pynvml.nvmlDeviceGetCount()
    except Exception:
        return local_rank
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        n_dev = len([v for v in vis.split(",") if v.strip()])
    if local_world <= 1 or n_dev <= local_world or n_dev % local_world or os.environ.get("DBEEL_NO_SPREAD"):
        return local_rank
    return local_rank * (n_dev // local_world)


def run_gpu(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = spread_device(int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    # Host placement first: the thread (and every thread torch / numpy start later) moves next to this rank's GPU, so the
    # pinned staging buffers allocated below are first-touched on the GPU's own NUMA node (main.rs:51-60 pins shards too).
    from dbeel_b200 import capi, sstable
    numa_node, numa_cpus = (-1, 0)
    if not os.environ.get("DBEEL_NO_NUMA_BIND"):
        numa_node, numa_cpus = capi.bind_to_gpu(local)
    import torch
    import torch.distributed as dist

    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            log(f"[bench] --gpus {args.gpus} needs torchrun with {args.gpus} ranks; running 1 GPU")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the compaction engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from dbeel_b200 import shard_jobs as sj
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.workload == "cfg5":
        import bench_cfg5
        return bench_cfg5.bench(args, torch, dist, dev, rank, world, local, ClockSampler, hbm_peak, METRIC, UNIT, log)
    # job hand-off (NCCL broadcast when N > 1): rank 0 owns the table; shard i's compaction runs on GPU i mod N
    n_jobs = N_JOBS if args.workload == "cfg2" else 1
    table = [sj.ShardJob(i, 40 + i, 8, 1_000_000, 256, False) for i in range(n_jobs)] if rank == 0 else None
    mine = sj.hand_off(table, dev)
    assert [j.shard_id % world for j in mine] == [rank] * len(mine), mine

    t = time.time()
    cfgs = [job_config(j, args.workload) for j in mine]
    jobs_runs = [make_runs_parallel(c) for c in cfgs]
    in_bytes_job = [sstable.input_bytes(r) for r in jobs_runs]
    in_bytes = sum(in_bytes_job)
    log(f"[bench r{rank}] numa node {numa_node} ({numa_cpus} cpus); generated {len(mine)} job(s) of {cfgs[0].name if cfgs else '-'}: "
        f"{in_bytes / 1e6:.1f} MB in {time.time() - t:.1f}s")

    eng = capi.Engine(local)
    keep = cfgs[0].keep_tombstones if cfgs else False
    opts = capi.make_opts(keep, seed=SEED32)
    bounds = [capi.compact_bound([(d.size, i.size) for d, i in runs], opts) for runs in jobs_runs]
    dc, ic, bc = (max(b[k] for b in bounds) for k in range(3)) if bounds else (0, 0, 0)

    # --overlap: two engines (two streams) take a GPU's jobs alternately.  Measured on B200: no gain (13.48 vs 13.59 ms for 8
    # jobs) -- every kernel of a job fills the GPU, and the block scheduler drains one grid before it starts the next
    # stream's, so two jobs' stages do not co-run.  Off by default; the rank's jobs run one after the other.
    n_eng = 2 if (len(mine) >= 2 and args.overlap) else 1
    engs = [eng] + [capi.Engine(local) for _ in range(n_eng - 1)]
    # device-resident inputs of every job of this rank; one output SSTable buffer set per engine, reused job after job --
    # with --dump-outputs one per job, so that every job's output of the last timed step is still there after it
    t_jobs = [[(torch.from_numpy(d).to(dev), torch.from_numpy(i).to(dev)) for d, i in runs] for runs in jobs_runs]
    slot = list(range(len(mine))) if args.dump_outputs else [j % n_eng for j in range(len(mine))]
    outs = [(torch.empty(dc + 64, dtype=torch.uint8, device=dev), torch.empty(ic + 64, dtype=torch.uint8, device=dev),
             torch.empty(bc + 64, dtype=torch.uint8, device=dev)) for _ in range(len(mine) if args.dump_outputs else n_eng)]
    d_jobs = [[(d.data_ptr(), d.numel(), i.data_ptr(), i.numel()) for d, i in t_runs] for t_runs in t_jobs]
    d_outs = [(od.data_ptr(), dc, oi.data_ptr(), ic, ob.data_ptr(), bc) for od, oi, ob in outs]
    ext = [torch.cuda.ExternalStream(e_.stream_ptr(), device=dev) for e_ in engs]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    KEYS = ("ms_total", "ms_extract", "ms_merge", "ms_resolve", "ms_gather", "kernel_launches", "gather_bytes", "input_bytes", "output_bytes")
    solo = {k: 0.0 for k in KEYS}

    # ---- (1) every job alone on the GPU: the per-job figures (ms_per_job, stage_ms, roofline of the gather kernel)
    solo_steps = max(1, min(3, args.steps))
    for rep in range(2 + solo_steps):
        for d_runs in d_jobs:
            eng.compact_device(d_runs, d_outs[0], opts)
            if rep >= 2:
                st = eng.stats()
                for k in KEYS:
                    solo[k] += st[k]
    solo_runs = solo_steps * len(d_jobs)

    # ---- (2) the timed region: K steps, each one pass over this rank's jobs, two in flight when there are two engines
    acc = {"kernel_launches": 0}
    lock = threading.Lock()
    last = [None] * len(d_jobs)  # (data_len, index_len, bloom_len, items) of every job in the latest step

    def worker(ei: int, record: bool):
        n_l = 0
        for j in range(ei, len(d_jobs), n_eng):
            last[j] = engs[ei].compact_device(d_jobs[j], d_outs[slot[j]], opts)
            if record:
                n_l += engs[ei].stats()["kernel_launches"]
        if record:
            with lock:
                acc["kernel_launches"] += n_l

    def step(record: bool) -> float:
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in engs]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in engs]
        for k in range(n_eng):
            ev0[k].record(ext[k])
        if n_eng == 1:
            worker(0, record)
        else:
            ths = [threading.Thread(target=worker, args=(k, record)) for k in range(n_eng)]
            for th in ths:
                th.start()
            for th in ths:
                th.join()
        for k in range(n_eng):
            ev1[k].record(ext[k])
        torch.cuda.synchronize()
        return max(a.elapsed_time(b) for a in ev0 for b in ev1)  # first start .. last end over the engines' streams

    for _ in range(max(3, args.warmup)):
        step(False)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        dev_ms += step(True)
    barrier()
    t1 = time.perf_counter()
    sampler.stop()
    wall_ms = (t1 - t0) * 1e3
    clocks = sampler.summary(t0, t1)
    if args.dump_outputs:
        for j, job in enumerate(mine):
            dl, il, bl, items = last[j]
            od, oi, ob = outs[slot[j]]
            dump_job_outputs(args.dump_outputs, job.shard_id, od[:dl], oi[:il], ob[:bl] if bl else None, items)

    # max over ranks of the device time (CUDA events on the engines' streams, summed over the K steps)
    tm = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device=dev)
    sums = torch.tensor([float(in_bytes), float(acc["kernel_launches"]), solo["ms_total"], solo["ms_extract"], solo["ms_merge"],
                         solo["ms_resolve"], solo["ms_gather"], float(solo["gather_bytes"]), float(solo["input_bytes"]),
                         float(solo["output_bytes"]), float(len(mine)), float(solo_runs)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    dev_ms_max, wall_ms_max = (float(x) for x in tm.tolist())
    (total_in, launches, s_total, s_extract, s_merge, s_resolve, s_gather, s_gbytes, s_in, s_out, jobs_all, job_runs) = (float(x) for x in sums.tolist())
    value = total_in * args.steps / 1e6 / (dev_ms_max / 1e3)

    # ---- end to end through the host entry point (pinned host buffers, H2D + D2H timed)
    del t_jobs, d_jobs, outs, d_outs, ext
    for e_ in engs[1:]:
        e_.close()
    torch.cuda.empty_cache()
    e2e_steps = max(2, min(3 if world == 1 else 5, args.steps))
    t = time.time()
    pins, h_jobs = [], []
    for runs in jobs_runs:
        h_runs = []
        for d, i in runs:
            pd, pi = capi.PinnedBuffer(d.size), capi.PinnedBuffer(i.size)
            pd.array[:] = d
            pi.array[:] = i
            pins += [pd, pi]
            h_runs.append((pd.array, pi.array))
        h_jobs.append(h_runs)
    pod, poi, pob = capi.PinnedBuffer(max(1, dc)), capi.PinnedBuffer(max(1, ic)), capi.PinnedBuffer(max(1, bc))
    log(f"[bench r{rank}] pinned {sum(p.nbytes for p in pins) / 1e9:.1f} GB of host input in {time.time() - t:.1f}s")
    out_bufs = (pod.array, poi.array, pob.array)
    hres = None
    for h_runs in h_jobs[:1]:
        hres = eng.compact(h_runs, keep, seed=SEED32, out_buffers=out_bufs)
    barrier()
    e0 = time.perf_counter()
    e2e_kernel_ms, e2e_parts = 0.0, 0
    for _ in range(e2e_steps):
        for h_runs in h_jobs:
            hres = eng.compact(h_runs, keep, seed=SEED32, out_buffers=out_bufs)
            e2e_kernel_ms += eng.stats()["ms_total"]
            e2e_parts = eng.stats()["partitions"]
    torch.cuda.synchronize()
    e_rank = (time.perf_counter() - e0) * 1e3  # this rank's own time, before the closing barrier
    barrier()
    e1 = time.perf_counter()
    out_bytes_job = int(hres[0].size + hres[1].size + (hres[2].size if hres[2] is not None else 0)) if hres else 0
    e2e_ms = torch.tensor([(e1 - e0) * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = total_in * e2e_steps / 1e6 / (float(e2e_ms[0]) / 1e3)
    # per-rank host-link rates (input + output bytes of the rank's jobs over its own e2e time)
    link = torch.zeros(world, dtype=torch.float64, device=dev)
    link[rank] = (in_bytes + out_bytes_job * len(mine)) * e2e_steps / 1e9 / (e_rank / 1e3) if e_rank > 0 else 0.0
    if world > 1:
        dist.all_reduce(link, op=dist.ReduceOp.SUM)

    # ---- byte parity of every job of every rank against the CPU oracle (outside the timed regions)
    cpu = None
    parity_mine = None
    if not args.no_cpu:
        import oracle
        from concurrent.futures import ThreadPoolExecutor
        t = time.perf_counter()
        first = oracle.compact(jobs_runs[0], keep, seed=SEED32, emulate_page_cache=True) if jobs_runs else None
        cpu_s = time.perf_counter() - t
        if rank == 0 and world == 1 and first is not None:
            cpu = {"value": round(in_bytes_job[0] / 1e6 / cpu_s, 2), "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": f"one full job of the workload ({cfgs[0].name}: {in_bytes_job[0] / 1e6:.0f} MB in, {cpu_s:.1f} s), 1 pass, "
                             "C oracle port of LSMTree::compact incl. page-cache write-through copies, RAM-resident files"}
        parity_mine = True
        with ThreadPoolExecutor(max_workers=max(1, min(len(jobs_runs), 8))) as ex:
            futs = [None] + [ex.submit(oracle.compact, r, keep, SEED32_DEFAULT_MIN, SEED32, True) for r in jobs_runs[1:]]
            for k, h_runs in enumerate(h_jobs):
                got = eng.compact(h_runs, keep, seed=SEED32, out_buffers=out_bufs)
                exp = first if k == 0 else futs[k].result()
                ok = same_output(got, exp)
                parity_mine = parity_mine and ok
                if not ok:
                    log(f"[bench r{rank}] job {mine[k].shard_id}: output differs from the oracle")
                futs[k] = None
        log(f"[bench r{rank}] byte parity of {len(h_jobs)} job(s) vs the oracle: {parity_mine} ({time.perf_counter() - t:.0f}s)")
    par = torch.tensor([1.0 if parity_mine in (True, None) else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(par, op=dist.ReduceOp.MIN)
    parity_all = None if args.no_cpu else bool(par[0] > 0.5)

    peak, peak_src = hbm_peak()
    others = None
    if rank == 0 and world == 1 and not args.no_cpu and args.workload == "cfg2" and not args.no_others:
        del pins, h_jobs, jobs_runs
        others = other_configs(eng, torch, dev, peak)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    ms_job = s_total / job_runs                       # mean CUDA-event ms of one compaction (configs[1] shape)
    g_ms = s_gather / job_runs
    gbytes = s_gbytes / job_runs
    achieved = gbytes / 1e9 / (g_ms / 1e3)
    algo_job = (s_in + s_out) / job_runs
    traffic, traffic_src = gather_traffic_from_profile()
    cfg_line = common_config() if args.workload == "cfg2" else {"workload": cfgs[0].name, "runs": cfgs[0].n_runs,
                                                                "keys_per_run": cfgs[0].keys_per_run, "doc_bytes": cfgs[0].doc_bytes,
                                                                "jobs": 1, "keep_tombstones": keep, "bloom": True}
    cfg_line.update({"jobs_per_gpu": len(mine), "input_bytes_per_step": int(total_in), "input_bytes_per_job": in_bytes_job[0] if in_bytes_job else 0,
                     "output_bytes_per_job": out_bytes_job,
                     "l2_policy": "inputs_larger_than_l2 (2.55 GB per job vs 126 MB L2)",
                     "parallelism": f"{int(jobs_all)} independent shard compactions over {world} GPU(s), shard i on GPU i mod N, no data-path collective",
                     "engines_per_gpu": n_eng,
                     "timing": "per step: CUDA events on the engines' streams, first start to last end of the rank's jobs (two jobs in flight "
                               "with --overlap); sum over the K steps, max over ranks.  ms_per_job / stage_ms / roofline: every job alone",
                     "host_placement": {"numa_node": numa_node, "cpus": numa_cpus, "rank0_gpu": local,
                                        "ranks_to_gpus": "rank r -> GPU r * n_gpus / N (spread over both CPU sockets)"}})
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": round(dev_ms_max / args.steps, 4), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": cfg_line,
        "wall_ms_per_step": round(wall_ms_max / args.steps, 4),
        "ms_per_job": round(ms_job, 4),
        "stage_ms": {"ms_extract": round(s_extract / job_runs, 4), "ms_merge": round(s_merge / job_runs, 4),
                     "ms_resolve": round(s_resolve / job_runs, 4), "ms_gather": round(g_ms, 4)},
        "pipeline_roofline": {"algo_bytes": int(algo_job), "achieved_gbs": round(algo_job / 1e9 / (ms_job / 1e3), 1),
                              "frac": round(algo_job / 1e9 / (ms_job / 1e3) / peak, 4),
                              "read_only_frac": round(s_in / job_runs / 1e9 / (ms_job / 1e3) / peak, 4),
                              "per": "one job (configs[1] shape) alone on the GPU, first to last kernel",
                              "frac_in_timed_region": round(algo_job * jobs_all * args.steps / 1e9 / (dev_ms_max / 1e3) / peak / world, 4)},
        "roofline": {"kernel": GATHER_KERNEL, "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                     "algo_bytes_per_launch": int(gbytes), "ms_per_launch": round(g_ms, 4), "peak_source": peak_src},
        "cpu_baseline": cpu,
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": int(total_in),
                "d2h_bytes_per_step": int(out_bytes_job * jobs_all), "steps": e2e_steps,
                "ms_per_step": round(float(e2e_ms[0]) / e2e_steps, 3),
                "ms_kernels_per_job": round(e2e_kernel_ms / max(1, e2e_steps * len(mine)), 3), "partitions": e2e_parts,
                "host_link_gbs_per_rank": [round(float(x), 1) for x in link.tolist()],
                "host_dma_ceiling_gbs_per_gpu": {"1_gpu": 91.4, "2_gpus_two_sockets": 91.9, "4_gpus_two_sockets": 77.9, "4_gpus_one_socket": 47.2,
                                                 "8_gpus": 47.3, "what": "plain cudaMemcpyAsync H2D + D2H at once, pinned NUMA-local memory, "
                                                 "cfg2-sized buffers, all listed GPUs at once", "source": "profiles/r02_pcie_topology.txt"},
                "api": "dbeel_compact (host pinned buffers; key-range partitions pipelined over H2D / kernels / D2H streams)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "parity_vs_oracle": parity_all,
        "parity_all_ranks": parity_all,
        "other_configs": others,
    }
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs, "jobs_rank0": [j.shard_id for j in mine],
                                "output_buffers": "one set per job, where a run without --dump-outputs reuses one set per engine: "
                                                  "the timed kernels wrote to other (and more) HBM than in such a run"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------ reference arm

def mem_available_bytes() -> int:
    try:
        with open("/proc/meminfo") as f:
            for ln in f:
                if ln.startswith("MemAvailable:"):
                    return int(ln.split()[1]) * 1024
    except Exception:
        pass
    return 64 << 30


def ref_jobs_per_step(threads: int, floor_threads: int, t_cal: float, steps: int, warm: int, budget_s: float) -> int:
    """Concurrent full-size jobs per step of the reference arm: `floor_threads` of them took t_cal seconds; at that (memory-
    bandwidth-bound) rate a step of n jobs takes n * t_cal / floor_threads, and steps + warm of them have to fit budget_s."""
    per_job_s = max(1e-3, t_cal / floor_threads)
    fit = int(budget_s / max(1, steps + warm) / per_job_s)
    return max(floor_threads, min(threads, fit))


def run_reference(args):
    """The reference's CPU implementation of the path on this box's host cores: the C oracle port of LSMTree::compact
    (the Rust reference cannot be built here: no cargo/rustc), one single-threaded FULL-SIZE shard compaction per core,
    all cores busy -- dbeel's thread-per-core model (main.rs:51-60) on the GPU arm's own config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from dbeel_b200 import sstable
    from dbeel_b200 import workloads as W

    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    steps, warm = args.steps, args.warmup
    # every thread compacts one full cfg2-shaped shard: ~2.1 GB of output + the reader / heap state, inputs shared
    # read-only between threads (8 distinct shards, 20 GB) -> budget 5 GB per thread
    distinct_n = min(N_JOBS, cores)
    budget = int(mem_available_bytes() * 0.6) - distinct_n * (3 << 30)
    threads = max(1, min(cores, 64, budget // (5 << 30)))
    t = time.time()
    distinct = [make_runs_parallel(W.cfg4_shard(i)) for i in range(distinct_n)]
    shards = [distinct[i % len(distinct)] for i in range(threads)]  # inputs are read-only: threads may share them
    in_bytes = sum(sstable.input_bytes(s) for s in shards)
    log(f"[bench ref] {threads} threads x one full cfg2-shaped compaction each ({in_bytes / 1e6:.0f} MB per step), "
        f"{distinct_n} distinct shards generated in {time.time() - t:.0f}s")

    kept = {}  # --dump-outputs: shard id -> (data, index, bloom | None, items) of the distinct shards in the last step

    def one(s, k=0, keep=False):
        out = oracle.compact(s, False, seed=SEED32, emulate_page_cache=True)
        if keep and k < distinct_n:
            kept[k] = out

    def step(keep=False):
        ts = [threading.Thread(target=one, args=(s, k, keep)) for k, s in enumerate(shards)]
        for th in ts:
            th.start()
        for th in ts:
            th.join()

    # The whole --steps K --warmup W run has to end within a few minutes (DBEEL_REF_BUDGET_S, default 210 s of stepping): a step
    # is `threads` concurrent FULL jobs, and 64 of them take ~38 s on this host (the path is memory-bandwidth-bound: 64 threads
    # deliver what ~8 do), so the number of concurrent jobs per step is cut to what fits -- never below the 8 jobs of one GPU
    # step.  Calibration: the step's own 8 jobs on 8 threads, untimed.
    budget_s = float(os.environ.get("DBEEL_REF_BUDGET_S", "210"))
    floor_threads = min(threads, N_JOBS)
    if threads > floor_threads:
        full = shards
        shards = full[:floor_threads]
        t_cal = time.perf_counter()
        step()
        t_cal = time.perf_counter() - t_cal
        threads = ref_jobs_per_step(threads, floor_threads, t_cal, steps, warm, budget_s)
        shards = full[:threads]
        in_bytes = sum(sstable.input_bytes(s) for s in shards)
        log(f"[bench ref] calibration: {floor_threads} concurrent jobs in {t_cal:.1f}s -> {threads} concurrent jobs per step "
            f"for {steps}+{warm} steps in ~{budget_s:.0f}s")
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for k in range(steps):
        step(keep=bool(args.dump_outputs) and k == steps - 1)
    dt = time.perf_counter() - t0
    value = in_bytes * steps / 1e6 / dt
    if args.dump_outputs:
        import torch
        for k, (d, i, b, n) in sorted(kept.items()):
            dump_job_outputs(args.dump_outputs, k, torch.from_numpy(d), torch.from_numpy(i), None if b is None else torch.from_numpy(b), n)
        dumped = sorted(kept)
        kept.clear()
        if len(dumped) < N_JOBS:
            log(f"[bench ref] --dump-outputs: wrote jobs {dumped} only, not all {N_JOBS}: the last step ran {threads} concurrent "
                f"jobs over {distinct_n} distinct shards")
    # secondary: one thread alone on the same shape (no memory-bandwidth sharing)
    t1 = time.perf_counter()
    one(shards[0])
    alone = sstable.input_bytes(shards[0]) / 1e6 / (time.perf_counter() - t1)
    sample = (f"{threads} concurrent single-threaded shard compactions per step (as many as fit {steps}+{warm} steps into ~{budget_s:.0f} s, at least "
              f"the {N_JOBS} jobs of one GPU step; the path is memory-bandwidth-bound beyond ~8 threads), each the FULL job of the GPU arm's config "
              f"(8 runs x 1,000,000 keys x 256 B docs, seeds 40+i; {in_bytes / 1e6:.0f} MB in per step), RAM-resident files, "
              "page-cache write-through copies emulated")
    cfg_line = common_config()
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": round(dt / steps * 1e3, 2), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": cfg_line, "threads": threads, "jobs_per_step": threads, "one_thread_alone_mbs": round(alone, 1),
            "cpu_baseline": {"value": round(value, 2), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": round(value, 2), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs, "jobs": dumped}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="dbeel_b200", choices=["dbeel_b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the oracle legs: cpu_baseline, byte parity, other_configs (profiling runs)")
    ap.add_argument("--overlap", action="store_true", help="two engines per GPU taking the rank's jobs alternately (measured: no gain)")
    ap.add_argument("--no-others", action="store_true", help="skip the other_configs block (cfg1 / cfg3 / cfg5-shard evidence)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg5"],
                    help="cfg2 (default): BASELINE.json's headline, 8 shard jobs of configs[1]'s shape; cfg5: configs[4]")
    ap.add_argument("--writes", type=int, default=0, help="cfg5: arrivals in the stream (default 32M)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what every job of the last step returned (length, seeded byte samples "
                         "and block sums of its .data / .index / .bloom) as DIR/job<i>_*.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload == "cfg5":
        ap.error("--dump-outputs covers the compaction jobs of the cfg2 / cfg3 workloads, not cfg5")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
