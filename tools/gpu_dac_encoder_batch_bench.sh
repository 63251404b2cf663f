#!/bin/bash
# DAC encoder batch benchmark (tools/dac_encoder_batch_bench.py) on one GPU: tools/gpu_dac_encoder_batch_bench.sh [OUT_DIR]
# The result lands in OUT_DIR/dac_encoder_batch_bench.json (default: bench_outputs/, which git ignores).
out="${1:-bench_outputs}"
mkdir -p "$out"
python tools/dac_encoder_batch_bench.py "$out/dac_encoder_batch_bench.json"
