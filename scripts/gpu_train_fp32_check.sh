#!/bin/bash
# Build, the fp32 training-route GPU tests, the rest of the GPU suite, smoke, the default bench line with --dump-outputs
# (compared file for file with the same line of a second, built checkout given as PARENT_TREE, e.g. the parent commit)
# and scripts/bench_fp32_train.py; logs and JSON lines go to OUTPUT_DIR (run from the repository root on a B200).
set -x
OUT=${1:?usage: scripts/gpu_train_fp32_check.sh OUTPUT_DIR [PARENT_TREE]}
PARENT=$2
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
python -c 'import __graft_entry__ as g; g.build()' > $OUT/build.log 2>&1 || { tail -20 $OUT/build.log; exit 1; }
timeout 1500 python -m pytest tests/test_loss_fp32_gpu.py -m gpu -q -s -rs --durations=8 > $OUT/pytest_fp32_train.log 2>&1; echo "pytest rc=$?" >> $OUT/pytest_fp32_train.log
grep -E "passed|failed|Error|assert|fp32|largest" $OUT/pytest_fp32_train.log | cut -c 1-400 | head -80
python -c 'import __graft_entry__ as g; g.smoke()' > $OUT/smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/smoke.log
tail -n 2 $OUT/smoke.log
timeout 1200 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs $OUT/dump_this > $OUT/bench_default.json 2> $OUT/bench_default.err
tail -c 600 $OUT/bench_default.json
if [ -n "$PARENT" ]; then
  (cd "$PARENT" && timeout 1200 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs $OUT/dump_parent) > $OUT/bench_parent.json 2> $OUT/bench_parent.err
  tail -c 600 $OUT/bench_parent.json
  python - "$OUT/dump_this" "$OUT/dump_parent" <<'PY' | tee $OUT/dump_compare.txt
import os, sys
import numpy as np
a, b = sys.argv[1], sys.argv[2]
fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
print("files", len(fa), len(fb), "same names" if fa == fb else "DIFFERENT names")
diff = [f for f in fa if f in fb and not np.array_equal(np.load(os.path.join(a, f)), np.load(os.path.join(b, f)))]
print("bitwise different:", diff if diff else "none")
PY
fi
timeout 900 python scripts/bench_fp32_train.py --steps 10 --warmup 3 --out $OUT/r11_fp32_train_bench_n1.jsonl > $OUT/bench_fp32_train.log 2>&1; echo "bench_fp32_train rc=$?"
cut -c 1-500 $OUT/bench_fp32_train.log | tail -20
timeout 2400 python -m pytest tests -m gpu -q --maxfail=20 --durations=12 --ignore=tests/test_loss_fp32_gpu.py > $OUT/pytest_gpu.log 2>&1; echo "pytest rc=$?" >> $OUT/pytest_gpu.log
tail -n 6 $OUT/pytest_gpu.log
