#!/bin/bash
# DAC decoder batch benchmark (tools/dac_batch_bench.py) on one GPU: tools/gpu_dac_batch_bench.sh [OUT_DIR]
# The result lands in OUT_DIR/dac_batch_bench.json (default: bench_outputs/, which git ignores).
out="${1:-bench_outputs}"
mkdir -p "$out"
python tools/dac_batch_bench.py "$out/dac_batch_bench.json"
