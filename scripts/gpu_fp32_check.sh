#!/bin/bash
# Build, the fp32-evaluation GPU tests (with their measurements printed), the whole GPU suite, smoke, the default bench
# line and scripts/bench_fp32_eval.py; logs and JSON lines go to the directory given as the only argument (run from the
# repository root on a B200).
set -x
OUT=${1:?usage: scripts/gpu_fp32_check.sh OUTPUT_DIR}
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > $OUT/fp32_build.log 2>&1 || { tail -20 $OUT/fp32_build.log; exit 1; }
timeout 1500 python -m pytest tests/test_fp32_eval_gpu.py -m gpu -q -s --durations=8 > $OUT/fp32_pytest_new.log 2>&1; echo "pytest rc=$?" >> $OUT/fp32_pytest_new.log
grep -E "^\[|passed|failed|Error|assert" $OUT/fp32_pytest_new.log | head -60
timeout 2400 python -m pytest tests -m gpu -q --maxfail=20 --durations=12 --ignore=tests/test_fp32_eval_gpu.py > $OUT/fp32_pytest_gpu.log 2>&1; echo "pytest rc=$?" >> $OUT/fp32_pytest_gpu.log
tail -n 6 $OUT/fp32_pytest_gpu.log
python -c 'import __graft_entry__ as g; g.smoke()' > $OUT/fp32_smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/fp32_smoke.log
tail -n 2 $OUT/fp32_smoke.log
timeout 1200 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/fp32_bench_default.json 2> $OUT/fp32_bench_default.err
tail -c 300 $OUT/fp32_bench_default.json
timeout 1500 python scripts/bench_fp32_eval.py --pairs 10500 100000 1000000 --width 1200 --csls-k 10 --steps 3 --warmup 1 > $OUT/fp32_bench.jsonl 2> $OUT/fp32_bench.err
cat $OUT/fp32_bench.jsonl | cut -c 1-900
tail -5 $OUT/fp32_bench.err
