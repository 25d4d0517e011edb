"""bench.py --dump-outputs: what dump_job_outputs writes for one compaction (the oracle's, at test scale) is reproducible,
sized as documented and accounts for every output byte; on the GPU, the files the GPU arm writes for job i are those of
job i's compaction."""
import argparse
import json
import os

import numpy as np
import pytest
import torch

import bench
import oracle
from dbeel_b200 import workloads as W


def test_dump_outputs_are_reproducible_and_cover_every_byte(tmp_path):
    runs = W.make_merge_runs(W.scaled(W.cfg4_shard(3), 20_000))
    d, i, b, n = oracle.compact(runs, False, seed=bench.SEED32)
    assert b is not None and d.size > bench.DUMP_SAMPLE["data"] and b.size < bench.DUMP_SAMPLE["bloom"]  # sampled and whole
    for k in range(2):
        bench.dump_job_outputs(str(tmp_path / f"run{k}"), 3, torch.from_numpy(d), torch.from_numpy(i), torch.from_numpy(b), n)
    names = sorted(os.listdir(tmp_path / "run0"))
    assert names == sorted(os.listdir(tmp_path / "run1")) and len(names) == 7
    for f in names:
        assert np.array_equal(np.load(tmp_path / "run0" / f), np.load(tmp_path / "run1" / f)), f

    got = {f[len("job3_"):-len(".npy")]: np.load(tmp_path / "run0" / f) for f in names}
    assert got["lengths"].tolist() == [d.size, i.size, b.size, n]
    for name, full in (("data", d), ("index", i), ("bloom", b)):
        sample, sums = got[f"{name}_sample"], got[f"{name}_blocksum"]
        assert sample.dtype == np.float32 and sample.size == min(full.size, bench.DUMP_SAMPLE[name])
        assert sums.dtype == np.float64 and sums.size == -(-full.size // bench.DUMP_BLOCK)
        assert sums.sum() == full.sum(dtype=np.int64) and sums[-1] == full[(sums.size - 1) * bench.DUMP_BLOCK:].sum()
    assert np.array_equal(got["bloom_sample"], b.astype(np.float32))

    bench.dump_job_outputs(str(tmp_path / "nobloom"), 0, torch.from_numpy(d), torch.from_numpy(i), None, n)
    assert np.load(tmp_path / "nobloom" / "job0_lengths.npy")[2] == 0
    assert np.load(tmp_path / "nobloom" / "job0_bloom_sample.npy").size == 0
    assert np.load(tmp_path / "nobloom" / "job0_bloom_blocksum.npy").size == 0


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, True])
def test_gpu_arm_dumps_what_every_job_computed(tmp_path, monkeypatch, capsys, overlap):
    """run_gpu with --dump-outputs, every job of the default workload scaled to 20k keys per run, one engine or two taking
    the jobs alternately: job i's files are those of the oracle's compaction of job i's runs."""
    small = lambda job, workload="cfg2": W.scaled(W.cfg4_shard(job.shard_id), 20_000)
    monkeypatch.setattr(bench, "job_config", small)
    monkeypatch.setenv("DBEEL_NO_NUMA_BIND", "1")
    args = argparse.Namespace(gpus=1, steps=2, warmup=0, workload="cfg2", overlap=overlap, no_cpu=True, no_others=True,
                              dump_outputs=str(tmp_path / "gpu"))
    bench.run_gpu(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["engines_per_gpu"] == (2 if overlap else 1)
    assert line["dump_outputs"]["jobs_rank0"] == list(range(bench.N_JOBS))
    for i in range(bench.N_JOBS):
        runs = bench.make_runs_parallel(small(argparse.Namespace(shard_id=i)))
        d, x, b, n = oracle.compact(runs, False, seed=bench.SEED32, emulate_page_cache=True)
        bench.dump_job_outputs(str(tmp_path / "oracle"), i, torch.from_numpy(d), torch.from_numpy(x),
                               None if b is None else torch.from_numpy(b), n)
    names = sorted(os.listdir(tmp_path / "oracle"))
    assert len(names) == 7 * bench.N_JOBS and names == sorted(os.listdir(tmp_path / "gpu"))
    for f in names:
        assert np.array_equal(np.load(tmp_path / "gpu" / f), np.load(tmp_path / "oracle" / f)), f
