#!/bin/bash
# Variable-length decode benchmark (tools/varlen_bench.py) on one GPU: tools/gpu_varlen_bench.sh [OUT_DIR]
# The result lands in OUT_DIR/varlen_bench.json (default: bench_outputs/, which git ignores).
out="${1:-bench_outputs}"
mkdir -p "$out"
python tools/varlen_bench.py "$out/varlen_bench.json"
