#!/bin/bash
# Forward kernels one by one against fp64 references (tests/test_gpu_fwd_kernels.py) with -s, and the largest value of
# every printed metric per test section and dtype, to be copied into the bound comments; which A/B switches and launch
# forms gave bit-identical outputs.  With `all`: also the rest of `pytest -m gpu`, smoke() and the default bench line.
# The file takes about 10 s on one B200.
# usage: fwd_kernels_check.sh OUT_DIR [all]
set -u
OUT=$(realpath -m "${1:?output directory}")
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/gpu.txt
python -m photoverse_b200.build > $OUT/build.log 2>&1 || { echo "build failed"; tail -30 $OUT/build.log; exit 1; }
timeout 600 python -m pytest tests/test_gpu_fwd_kernels.py -q -s -m gpu -p no:cacheprovider > $OUT/fwd_pytest.log 2>&1
echo "fwd pytest rc=$?"; grep -E "^(FAILED|ERROR)|passed|failed" $OUT/fwd_pytest.log | tail -40
python - "$OUT/fwd_pytest.log" > $OUT/fwd_maxima.txt <<'PY'
import collections, re, sys
worst = collections.defaultdict(float)
where = {}
ident = collections.Counter()
for line in open(sys.argv[1]):
    m = re.match(r"\[(fwd:[^\]]+)\] (.*)", line)
    if not m:
        continue
    tag, rest = m.groups()
    if "identical" in tag:
        ident[(tag, re.sub(r"^\S+ \S+ \S+ ?", "", rest.split(":", 1)[1]).strip())] += 1
        continue
    for k, v in re.findall(r"(\w+)=([-+0-9.eE]+|inf|nan)(?=\s|$| of| ulp)", rest.split(":", 1)[-1]):
        try:
            x = float(v)
        except ValueError:
            continue
        if x >= worst[(tag, k)]:
            worst[(tag, k)], where[(tag, k)] = x, rest.split(":", 1)[0]
    for v, k in re.findall(r"([0-9.eE+-]+) (of the bound|ulp)", rest):
        if float(v) >= worst[(tag, k)]:
            worst[(tag, k)], where[(tag, k)] = float(v), rest.split(":", 1)[0]
for (tag, k), v in sorted(worst.items()):
    print(f"{tag:28s} {k:14s} {v:.3e}   at {where[(tag, k)]}")
for (tag, what), n in sorted(ident.items()):
    print(f"{tag:28s} {n:4d} x {what}")
PY
cat $OUT/fwd_maxima.txt
if [ "${2:-}" = "all" ]; then
  timeout 2400 python -m pytest tests -q -m gpu -p no:cacheprovider --ignore=tests/test_gpu_fwd_kernels.py > $OUT/gpu_pytest.log 2>&1
  echo "gpu pytest rc=$?"; tail -15 $OUT/gpu_pytest.log
  timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1
  echo "smoke rc=$?"; tail -3 $OUT/smoke.log
  timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 > $OUT/bench.log 2>&1
  echo "bench rc=$?"; tail -2 $OUT/bench.log | cut -c1-600
fi
