#!/bin/bash
# float32 models under torch.autocast: their GPU tests, the conversion / processor / training-step timing
# (tools/autocast_bench.py), smoke(), the default bench line and the rest of `pytest -m gpu`
# usage: autocast_check.sh OUT_DIR
set -u
OUT=${1:?output directory}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/gpu.txt
python -m photoverse_b200.build > $OUT/build.log 2>&1 || { echo "build failed"; tail -30 $OUT/build.log; exit 1; }
timeout 1500 python -m pytest tests/test_gpu_autocast.py -q -s > $OUT/autocast_pytest.log 2>&1
echo "autocast pytest rc=$?"; grep -E "cosine|passed|failed|Error|assert" $OUT/autocast_pytest.log | tail -40
timeout 900 python tools/autocast_bench.py --out $OUT/autocast_bench.json 2>&1 | tail -14
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -3 $OUT/smoke.log
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 > $OUT/bench.log 2>&1
echo "bench rc=$?"; tail -2 $OUT/bench.log | cut -c1-600
timeout 2400 python -m pytest tests -q -m gpu --ignore=tests/test_gpu_autocast.py > $OUT/gpu_pytest.log 2>&1
echo "gpu pytest rc=$?"; tail -15 $OUT/gpu_pytest.log
