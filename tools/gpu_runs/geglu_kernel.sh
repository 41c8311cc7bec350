#!/bin/bash
# GEGLU linear (ops.linear_geglu): parity tests, the backbone tests (exact native launch count), per-shape timing
# usage: geglu_kernel.sh OUT_DIR
set -u
OUT=${1:?output directory}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
timeout 1200 python -m pytest tests/test_gpu_geglu_linear.py tests/test_gpu_backbone.py -q > $OUT/geglu_pytest.log 2>&1
echo "pytest rc=$?"; tail -25 $OUT/geglu_pytest.log
timeout 600 python tools/geglu_bench.py --out $OUT/geglu_bench.json 2>&1 | tail -8
