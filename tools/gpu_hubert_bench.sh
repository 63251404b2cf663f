#!/bin/bash
# HuBERT semantic tokenizer benchmark (tools/hubert_bench.py) on one GPU: tools/gpu_hubert_bench.sh [OUT_DIR]
# The result lands in OUT_DIR/hubert_bench_b200.json (default: bench_outputs/, which git ignores).
out="${1:-bench_outputs}"
mkdir -p "$out"
python tools/hubert_bench.py "$out/hubert_bench_b200.json"
