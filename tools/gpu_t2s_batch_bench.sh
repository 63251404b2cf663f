#!/bin/bash
# Batched text-to-semantic decode benchmark (tools/t2s_batch_bench.py) on one GPU: tools/gpu_t2s_batch_bench.sh [OUT_DIR]
# The result lands in OUT_DIR/t2s_batch_bench.json (default: bench_outputs/, which git ignores).
out="${1:-bench_outputs}"
mkdir -p "$out"
python tools/t2s_batch_bench.py "$out/t2s_batch_bench.json"
