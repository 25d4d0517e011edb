#!/bin/bash
# Hash-range scan benchmark + the headline bench.py number in one run on a GPU machine.
# usage: tools/gpu_scan.sh [OUT_DIR] [scan_bench.py args]   (OUT_DIR default: a fresh temporary directory)
#   OUT_DIR/r03_scan_bench.json  tools/scan_bench.py's record (profiles/r03_scan_bench.json is a copy of one)
#   OUT_DIR/scan_bench.txt, OUT_DIR/bench_after_scan.txt, OUT_DIR/build.txt  the logs, bench.py's JSON line
out=${1:-$(mktemp -d)}
shift
mkdir -p "$out"
echo "writing to $out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
python -c "import __graft_entry__ as g; g.build()" > "$out/build.txt" 2>&1 || { tail -20 "$out/build.txt"; exit 1; }
timeout 1200 python tools/scan_bench.py --out "$out/r03_scan_bench.json" "$@" 2>&1 | tee "$out/scan_bench.txt"
timeout 1200 python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -2 | tee "$out/bench_after_scan.txt"
