#!/bin/bash
# End-to-end A/B of the fused GEGLU projection on one box: the unchanged bench.py, alternately from the parent commit's
# build (a `git archive` export with its library built, in the untracked directory MAIN_DIR) and from this tree, 3 runs
# each, latents dumped for comparison; then one training-step record per build.
# usage: geglu_ab.sh OUT_DIR MAIN_DIR
set -u
OUT=$(realpath -m "${1:?output directory}")
MAIN=${2:?directory of the previous build}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/gpu.txt
ARGS="--no-train-leg --no-cpu-baseline --no-cfg3-leg"
for i in 1 2 3; do
  (cd $MAIN && timeout 900 python bench.py $ARGS --dump-outputs $OUT/main_$i > $OUT/main_$i.json 2> $OUT/main_$i.err); echo "main $i rc=$?"
  timeout 900 python bench.py $ARGS --dump-outputs $OUT/branch_$i > $OUT/branch_$i.json 2> $OUT/branch_$i.err; echo "branch $i rc=$?"
done
(cd $MAIN && timeout 900 python bench.py --workload train --no-cpu-baseline > $OUT/train_main.json 2> $OUT/train_main.err); echo "train main rc=$?"
timeout 900 python bench.py --workload train --no-cpu-baseline > $OUT/train_branch.json 2> $OUT/train_branch.err; echo "train branch rc=$?"
python - "$OUT" <<'PY'
import json, statistics, sys, numpy as np
O = sys.argv[1]
def rec(p):
    for line in open(p):
        line = line.strip()
        if line.startswith("{"):
            return json.loads(line)
res = {}
for arm in ("main", "branch"):
    rs = [rec(f"{O}/{arm}_{i}.json") for i in (1, 2, 3)]
    res[arm] = [r["value"] for r in rs]
    for i, r in enumerate(rs, 1):
        print(arm, i, "value", r["value"], "clocks", json.dumps(r.get("clocks"))[:400])
mm, mb = statistics.median(res["main"]), statistics.median(res["branch"])
print("median main", mm, "branch", mb, "ratio", round(mb / mm, 4), "every branch > every main", min(res["branch"]) > max(res["main"]))
lat = {k: np.load(f"{O}/{k}/latents.npy").astype(np.float64) for k in ["main_1", "main_2", "main_3", "branch_1", "branch_2", "branch_3"]}
def d(a, b):
    x = lat[a] - lat[b]
    return float(np.sqrt((x ** 2).mean())), float(np.abs(x).max())
print("latent rms", float(np.sqrt((lat["main_1"] ** 2).mean())))
for a, b in [("main_1", "main_2"), ("main_1", "main_3"), ("main_2", "main_3"), ("branch_1", "main_1"), ("branch_2", "main_2"),
             ("branch_3", "main_3"), ("branch_1", "branch_2")]:
    print(f"{a} vs {b}: rms diff {d(a, b)[0]:.4f} max diff {d(a, b)[1]:.4f}")
for arm in ("main", "branch"):
    r = rec(f"{O}/train_{arm}.json")
    print("train", arm, "value", r.get("value"), r.get("unit"), "clocks", json.dumps(r.get("clocks"))[:300])
PY
