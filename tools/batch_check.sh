#!/bin/bash
# Batched generation on one B200, in one go: its GPU tests, the whole GPU suite, smoke(), a bench.py N=1 line and tools/batch_bench.py.
# Usage: tools/batch_check.sh <output directory>   (logs, the bench line and the batch_bench JSON are written there)
cd "$(dirname "$0")/.." || exit 1
OUT=${1:?usage: tools/batch_check.sh <output directory>}
mkdir -p "$OUT"
export BARK_B200_QUIET=1
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1 || { tail -40 "$OUT/build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.txt" 2>&1
timeout 1200 python -m pytest -q tests/test_batch_gpu.py > "$OUT/pytest_batch.log" 2>&1; echo "batch tests exit $?"
tail -25 "$OUT/pytest_batch.log"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/bench_n1.json" 2> "$OUT/bench_n1.err"; echo "bench exit $?"
tail -c 1500 "$OUT/bench_n1.json"
timeout 1200 python tools/batch_bench.py --out "$OUT/r03_batch_small_f16.json" > /dev/null 2> "$OUT/batch_bench.err"; echo "batch_bench exit $?"
tail -c 3000 "$OUT/batch_bench.err"
timeout 1500 python -m pytest -q -m gpu tests > "$OUT/pytest_gpu.log" 2>&1; echo "gpu suite exit $?"
tail -5 "$OUT/pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke exit $?"; tail -3 "$OUT/smoke.log"
