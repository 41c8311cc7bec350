#!/bin/bash
# LoRA on attn2.to_out.0: its GPU tests, smoke(), the q/k/v vs q/k/v/out training-step and generation timing
# (tools/lora_out_bench.py), and the q/k/v-only training step of bench.py alternately from the parent commit's build (a
# `git archive` export with its library built, in the untracked directory PARENT_DIR) and from this tree, 3 runs each.
# usage: lora_out_check.sh OUT_DIR PARENT_DIR
set -u
OUT=$(realpath -m "${1:?output directory}")
PARENT=${2:?directory of the parent build}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/gpu.txt
python -m photoverse_b200.build > $OUT/build.log 2>&1 || { echo "build failed"; tail -30 $OUT/build.log; exit 1; }
timeout 1200 python -m pytest tests/test_gpu_lora_out.py -q -s > $OUT/lora_out_pytest.log 2>&1
echo "lora_out pytest rc=$?"; grep -E "cosine|passed|failed|Error|assert" $OUT/lora_out_pytest.log | tail -30
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -3 $OUT/smoke.log
timeout 1200 python tools/lora_out_bench.py --out $OUT/lora_out_bench.json > $OUT/lora_out_bench.log 2>&1
echo "lora_out_bench rc=$?"; tail -4 $OUT/lora_out_bench.log | cut -c1-700
ARGS="--workload train --no-cpu-baseline --steps 10 --warmup 3"
for i in 1 2 3; do
  (cd $PARENT && timeout 600 python bench.py $ARGS > $OUT/train_parent_$i.json 2> $OUT/train_parent_$i.err); echo "train parent $i rc=$?"
  timeout 600 python bench.py $ARGS > $OUT/train_branch_$i.json 2> $OUT/train_branch_$i.err; echo "train branch $i rc=$?"
done
python - "$OUT" <<'PY'
import json, sys
O = sys.argv[1]
for arm in ("parent", "branch"):
    for i in (1, 2, 3):
        for line in open(f"{O}/train_{arm}_{i}.json"):
            if line.startswith("{"):
                r = json.loads(line)
                print("train", arm, i, "ms_per_step", r.get("ms_per_step"), "final_loss", r.get("final_loss"),
                      "launches", r.get("gpu_launches"))
PY
