#!/bin/bash
# Streamed hash-range scans on a GPU machine: every GPU test (old and new), the file-fed scan benchmark, then bench.py.
# usage: tools/gpu_scan_stream.sh OUT_DIR [scan_stream_bench.py args]
#   OUT_DIR/build.txt, OUT_DIR/pytest_gpu.txt            the build log, the GPU test run
#   OUT_DIR/r04_scan_stream.json, OUT_DIR/scan_stream_bench.txt   tools/scan_stream_bench.py's record (profiles/ holds a copy)
#   OUT_DIR/bench_after_scan_stream.txt                   bench.py's JSON line
out=${1:?usage: tools/gpu_scan_stream.sh OUT_DIR}
shift
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$out/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" > "$out/build.txt" 2>&1 || { tail -20 "$out/build.txt"; exit 1; }
timeout 1800 python -m pytest -q -m gpu tests 2>&1 | tail -30 | tee "$out/pytest_gpu.txt"
timeout 1200 python tools/scan_stream_bench.py --out "$out/r04_scan_stream.json" "$@" 2>&1 | tee "$out/scan_stream_bench.txt"
timeout 1200 python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -2 | tee "$out/bench_after_scan_stream.txt"
