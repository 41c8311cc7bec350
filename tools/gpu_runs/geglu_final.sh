#!/bin/bash
# With the fused GEGLU projection: the GPU suite (test_gpu_backbone.py and test_gpu_geglu_linear.py are run by
# geglu_kernel.sh), smoke(), and the kernel list of one UNet evaluation (profiles/unet_eval_kernels_r03.txt)
# usage: geglu_final.sh OUT_DIR
set -u
OUT=${1:?output directory}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
timeout 420 python -m pytest tests -m gpu -q --ignore=tests/test_gpu_backbone.py --ignore=tests/test_gpu_geglu_linear.py > $OUT/final_pytest.log 2>&1
echo "pytest rc=$?"; tail -12 $OUT/final_pytest.log
timeout 120 python __graft_entry__.py smoke > $OUT/final_smoke.log 2>&1; echo "smoke rc=$?"; tail -3 $OUT/final_smoke.log
(echo "== stock PyTorch epilogues (bench.py --stock-epilogues) =="; timeout 100 python tools/unet_profile.py --stock-epilogues --top 30 2>&1 | grep -v Warn | grep -v _warn;
 echo; echo "== pv_backbone.cu epilogues and the fused GEGLU projection (default) =="; timeout 100 python tools/unet_profile.py --top 30 2>&1 | grep -v Warn | grep -v _warn) > $OUT/unet_eval_kernels_r03.txt
echo "unet kernel lists rc=$?"
