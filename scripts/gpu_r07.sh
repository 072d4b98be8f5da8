#!/bin/bash
# Quotient polynomial: build, the new tests/test_gpu_quotient.py, the rest of the GPU suite, smoke, scripts/bench_quotient.py
# (2^16 range_check instances, domain 2^25) twice for the spread with its kernel table, scripts/bench_ntt.py at 2^26 and the flagship bench.
# Usage: scripts/gpu_r07.sh TAG OUTPUT_DIR
TAG=${1:?run tag}
OUT=${2:?output directory}; mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${TAG}_gpu.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/${TAG}_build.log 2>&1; echo "build exit $?"
timeout 1800 python -m pytest tests/test_gpu_quotient.py -q -m gpu > $OUT/${TAG}_pytest_quotient.log 2>&1; echo "pytest quotient exit $?"; tail -4 $OUT/${TAG}_pytest_quotient.log
timeout 1200 python -m pytest tests -q -m gpu --ignore=tests/test_gpu_quotient.py > $OUT/${TAG}_pytest_rest.log 2>&1; echo "pytest rest exit $?"; tail -2 $OUT/${TAG}_pytest_rest.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${TAG}_smoke.log 2>&1; echo "smoke exit $?"; tail -2 $OUT/${TAG}_smoke.log
for rep in 1 2; do
  timeout 600 python scripts/bench_quotient.py --trace-dir $OUT/${TAG}_trace$rep > $OUT/${TAG}_bench_quotient_$rep.json 2> $OUT/${TAG}_bench_quotient_$rep.err; echo "bench_quotient exit $?"; cat $OUT/${TAG}_bench_quotient_$rep.json; tail -3 $OUT/${TAG}_bench_quotient_$rep.err
done
timeout 600 python scripts/bench_ntt.py 26 > $OUT/${TAG}_ntt.jsonl 2> $OUT/${TAG}_ntt.err; echo "bench_ntt exit $?"; cut -c1-300 $OUT/${TAG}_ntt.jsonl
timeout 300 python bench.py --gpus 1 --steps 4 --warmup 3 > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err; echo "bench exit $?"; cut -c1-300 $OUT/${TAG}_bench.json
