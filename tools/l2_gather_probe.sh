#!/bin/bash
# Build and run the L2 gather-rate probe (no torch needed): tools/l2_gather_probe.sh [out.json]
set -e
bin=$(mktemp -d)/l2_gather_probe
/usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o "$bin" "$(dirname "$0")/l2_gather_probe.cu"
"$bin" | tee "${1:-/dev/null}"
rm -rf "$(dirname "$bin")"
