#!/bin/bash
# Regional identity masks (ip_adapter_masks): the new GPU tests, the whole GPU suite, smoke(), bench.py, and the per-call /
# per-generation cost of a mask (tools/ip_mask_bench.py -> OUT_DIR/ip_mask_bench.json).
# usage: ip_mask_check.sh OUT_DIR
set -u
OUT=$(realpath -m "${1:?output directory}")
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1 || { echo "build failed"; tail -30 $OUT/build.log; exit 1; }
timeout 1500 python -m pytest tests/test_gpu_ip_mask.py -q -s > $OUT/ip_mask_pytest.log 2>&1
echo "ip_mask pytest rc=$?"; grep -E "cosine|passed|failed|Error|assert" $OUT/ip_mask_pytest.log | tail -30
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -3 $OUT/smoke.log
timeout 900 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/bench.json 2> $OUT/bench.err
echo "bench rc=$?"; tail -1 $OUT/bench.json | cut -c1-600
timeout 900 python tools/ip_mask_bench.py --out $OUT/ip_mask_bench.json > $OUT/ip_mask_bench.log 2>&1
echo "ip_mask_bench rc=$?"; tail -12 $OUT/ip_mask_bench.log | cut -c1-400
timeout 2400 python -m pytest tests -q -m gpu --ignore=tests/test_gpu_ip_mask.py > $OUT/gpu_suite.log 2>&1
echo "gpu suite rc=$?"; grep -E "passed|failed|Error" $OUT/gpu_suite.log | tail -20
