#!/bin/bash
# Build, the fp32 link-search GPU tests, scripts/bench_fp32_links.py, the rest of the GPU suite, smoke and the default
# bench line; logs and JSON lines go to the directory given as the only argument (run from the repository root on a B200).
set -x
OUT=${1:?usage: scripts/gpu_links_check.sh OUTPUT_DIR}
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > $OUT/links_build.log 2>&1 || { tail -20 $OUT/links_build.log; exit 1; }
timeout 1200 python -m pytest tests/test_fp32_links_gpu.py -m gpu -q -rs --durations=8 > $OUT/links_pytest_new.log 2>&1; echo "pytest rc=$?" >> $OUT/links_pytest_new.log
grep -E "passed|failed|Error|assert|SKIP" $OUT/links_pytest_new.log | head -40
timeout 900 python scripts/bench_fp32_links.py --steps 5 --warmup 1 > $OUT/links_bench.jsonl 2> $OUT/links_bench.err
cut -c 1-600 $OUT/links_bench.jsonl
tail -5 $OUT/links_bench.err
timeout 2400 python -m pytest tests -m gpu -q --maxfail=20 --durations=12 --ignore=tests/test_fp32_links_gpu.py > $OUT/links_pytest_gpu.log 2>&1; echo "pytest rc=$?" >> $OUT/links_pytest_gpu.log
tail -n 6 $OUT/links_pytest_gpu.log
python -c 'import __graft_entry__ as g; g.smoke()' > $OUT/links_smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/links_smoke.log
tail -n 2 $OUT/links_smoke.log
timeout 1200 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/links_bench_default.json 2> $OUT/links_bench_default.err
tail -c 400 $OUT/links_bench_default.json
