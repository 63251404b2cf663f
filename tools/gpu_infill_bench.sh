#!/bin/bash
# S2A infilling benchmark (tools/infill_bench.py) on one GPU: tools/gpu_infill_bench.sh [OUT_DIR]
# The result lands in OUT_DIR/infill_bench_b200.json (default: bench_outputs/, which git ignores).
out="${1:-bench_outputs}"
mkdir -p "$out"
python tools/infill_bench.py "$out/infill_bench_b200.json"
