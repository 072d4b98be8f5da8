#!/bin/bash
# Openings (prover rounds 4 and 5): build, the new tests/test_gpu_openings.py, the rest of the GPU suite, smoke,
# scripts/bench_openings.py (2^16 range_check instances, domain 2^25) twice for the spread with its kernel table, and the flagship bench.
# Usage: scripts/gpu_r08.sh TAG OUTPUT_DIR
TAG=${1:?run tag}
OUT=${2:?output directory}; mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${TAG}_gpu.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/${TAG}_build.log 2>&1; echo "build exit $?"
timeout 1800 python -m pytest tests/test_gpu_openings.py -q -m gpu > $OUT/${TAG}_pytest_openings.log 2>&1; echo "pytest openings exit $?"; tail -4 $OUT/${TAG}_pytest_openings.log
for rep in 1 2; do
  timeout 600 python scripts/bench_openings.py --trace-dir $OUT/${TAG}_trace$rep > $OUT/${TAG}_bench_openings_$rep.json 2> $OUT/${TAG}_bench_openings_$rep.err; echo "bench_openings exit $?"; cat $OUT/${TAG}_bench_openings_$rep.json; tail -3 $OUT/${TAG}_bench_openings_$rep.err
done
timeout 300 python bench.py --gpus 1 --steps 4 --warmup 3 > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err; echo "bench exit $?"; cut -c1-300 $OUT/${TAG}_bench.json
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${TAG}_smoke.log 2>&1; echo "smoke exit $?"; tail -2 $OUT/${TAG}_smoke.log
timeout 1500 python -m pytest tests -q -m gpu --ignore=tests/test_gpu_openings.py > $OUT/${TAG}_pytest_rest.log 2>&1; echo "pytest rest exit $?"; tail -2 $OUT/${TAG}_pytest_rest.log
