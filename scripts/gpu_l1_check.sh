#!/bin/bash
# Build, GPU suite, smoke, default bench line and the --distance 1 measurements of scripts/bench_l1.py; logs and JSON
# lines go to the directory given as the only argument (run from the repository root on a B200).
set -x
OUT=${1:?usage: scripts/gpu_l1_check.sh OUTPUT_DIR}
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > $OUT/l1_build.log 2>&1 || { tail -20 $OUT/l1_build.log; exit 1; }
timeout 2400 python -m pytest tests -m gpu -q --maxfail=20 --durations=12 > $OUT/l1_pytest_gpu.log 2>&1; echo "pytest rc=$?" >> $OUT/l1_pytest_gpu.log
tail -n 20 $OUT/l1_pytest_gpu.log
python -c 'import __graft_entry__ as g; g.smoke()' > $OUT/l1_smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/l1_smoke.log
tail -n 3 $OUT/l1_smoke.log
timeout 1200 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/l1_bench_default.json 2> $OUT/l1_bench_default.err
tail -c 400 $OUT/l1_bench_default.json
for k in 10 3; do
  timeout 900 python scripts/bench_l1.py --pairs 10500 --width 1200 --csls-k $k --steps 20 --warmup 3 >> $OUT/l1_bench.jsonl
done
timeout 900 python scripts/bench_l1.py --pairs 10500 --width 1200 --nocsls --steps 20 --warmup 3 >> $OUT/l1_bench.jsonl
timeout 1200 python scripts/bench_l1.py --pairs 100000 --width 1200 --csls-k 10 --steps 5 --warmup 1 >> $OUT/l1_bench.jsonl
timeout 1200 torchrun --standalone --nproc-per-node 1 scripts/bench_l1.py --pairs 262144 --width 1200 --csls-k 10 --steps 2 --warmup 1 \
  --no-materialised >> $OUT/l1_bench.jsonl
cat $OUT/l1_bench.jsonl
