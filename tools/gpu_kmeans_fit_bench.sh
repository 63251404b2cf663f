#!/bin/bash
# K-means fit benchmark (tools/kmeans_fit_bench.py) on one GPU: tools/gpu_kmeans_fit_bench.sh [OUT_DIR]
# The result lands in OUT_DIR/kmeans_fit_bench_b200.json (default: bench_outputs/, which git ignores).
out="${1:-bench_outputs}"
mkdir -p "$out"
python tools/kmeans_fit_bench.py "$out/kmeans_fit_bench_b200.json"
