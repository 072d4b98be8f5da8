#!/bin/bash
# Lagrange-basis SRS from the monomial powers: build, the new tests/test_gpu_srs_lagrange.py, scripts/bench_srs_lagrange.py
# (2^16 .. 2^25, then the headline commitments), smoke, the flagship bench and the rest of the GPU suite.
# Usage: scripts/gpu_r09.sh TAG OUTPUT_DIR [rest]   ("rest": the existing GPU suite too)
TAG=${1:?run tag}
OUT=${2:?output directory}; mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${TAG}_gpu.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/${TAG}_build.log 2>&1; echo "build exit $?"
timeout 900 python -m pytest tests/test_gpu_srs_lagrange.py -q -m gpu --durations=20 > $OUT/${TAG}_pytest_srs_lagrange.log 2>&1; echo "pytest srs_lagrange exit $?"; tail -25 $OUT/${TAG}_pytest_srs_lagrange.log
timeout 900 python scripts/bench_srs_lagrange.py > $OUT/${TAG}_bench_srs_lagrange.json 2> $OUT/${TAG}_bench_srs_lagrange.err; echo "bench_srs_lagrange exit $?"; cat $OUT/${TAG}_bench_srs_lagrange.json; tail -6 $OUT/${TAG}_bench_srs_lagrange.err
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${TAG}_smoke.log 2>&1; echo "smoke exit $?"; tail -2 $OUT/${TAG}_smoke.log
timeout 300 python bench.py --gpus 1 --steps 4 --warmup 3 > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err; echo "bench exit $?"; cut -c1-300 $OUT/${TAG}_bench.json
if [ "$3" = rest ]; then
  timeout 1500 python -m pytest tests -q -m gpu --ignore=tests/test_gpu_srs_lagrange.py > $OUT/${TAG}_pytest_rest.log 2>&1; echo "pytest rest exit $?"; tail -4 $OUT/${TAG}_pytest_rest.log
fi
