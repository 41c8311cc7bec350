#!/bin/bash
# float16 inference path: its GPU tests, the rest of `pytest -m gpu`, smoke(), the default bench line and the fp16 / bf16
# processor timing (tools/f16_bench.py)
# usage: f16_check.sh OUT_DIR
set -u
OUT=${1:?output directory}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/gpu.txt
python -m photoverse_b200.build > $OUT/build.log 2>&1 || { echo "build failed"; tail -30 $OUT/build.log; exit 1; }
timeout 1500 python -m pytest tests/test_gpu_f16.py -q -s > $OUT/f16_pytest.log 2>&1
echo "f16 pytest rc=$?"; grep -E "max-abs|cosine|passed|failed|Error" $OUT/f16_pytest.log | tail -40
timeout 900 python tools/f16_bench.py --out $OUT/f16_bench.json 2>&1 | tail -8
timeout 2400 python -m pytest tests -q -m gpu > $OUT/gpu_pytest.log 2>&1
echo "gpu pytest rc=$?"; tail -15 $OUT/gpu_pytest.log
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -3 $OUT/smoke.log
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 > $OUT/bench.log 2>&1
echo "bench rc=$?"; tail -2 $OUT/bench.log | cut -c1-600
