#!/bin/bash
# Tensor-core selector products in the generic gate check (k_check_tc), against the parent tree on the same B200: bench.py (default arguments) alternated three
# times per tree with kernel_ms.check and the clock sample of every run, bench.py --dump-outputs of both trees compared file by file,
# then smoke and the whole GPU suite on this tree.
# Usage: scripts/gpu_r11.sh TAG OUTPUT_DIR PARENT_TREE STAGE   (PARENT_TREE: a checkout of the parent commit, both trees built;
#        STAGE: bench | outputs | tests [test files, default tests/] -- one stage per call keeps each call short)
TAG=${1:?run tag}; OUT=${2:?output directory}; PAR=${3:?parent tree}; STAGE=${4:?bench, outputs or tests}
mkdir -p $OUT; OUT=$(cd $OUT && pwd); PAR=$(cd $PAR && pwd); NEW=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/${TAG}_gpu.txt 2>&1; cat $OUT/${TAG}_gpu.txt
(python -c "import __graft_entry__ as g; g.build()" > $OUT/${TAG}_build.log 2>&1; echo "build exit $?") &
(cd $PAR && python -c "import __graft_entry__ as g; g.build()" > $OUT/${TAG}_build_parent.log 2>&1; echo "parent build exit $?") &
wait
summary() { python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); c=d.get('clocks') or {}
print(sys.argv[2], round(d['value']/1e9,4), 'G/s', 'step', round(d['ms_per_step'],2), 'ms', 'check', round(d['kernel_ms']['check'],2), 'ms', 'clocks', json.dumps(c)[:200])" $1 $2; }
if [ $STAGE = bench ]; then
for rep in 1 2 3; do
  for tree in parent new; do
    dir=$NEW; [ $tree = parent ] && dir=$PAR
    (cd $dir && timeout 600 python bench.py > $OUT/${TAG}_bench_${tree}_$rep.json 2> $OUT/${TAG}_bench_${tree}_$rep.err); echo "bench $tree $rep exit $?"
    summary $OUT/${TAG}_bench_${tree}_$rep.json "$tree $rep"
  done
done
fi
if [ $STAGE = outputs ]; then
DUMP=$(mktemp -d)
for tree in parent new; do
  dir=$NEW; [ $tree = parent ] && dir=$PAR
  (cd $dir && timeout 600 python bench.py --dump-outputs $DUMP/$tree > $OUT/${TAG}_dump_${tree}.json 2> $OUT/${TAG}_dump_${tree}.err); echo "dump $tree exit $?"
done
(cd $DUMP/parent && for f in *.npy; do if cmp -s $f ../new/$f; then echo "identical $f $(sha256sum < $f | cut -c1-16)"; else echo "DIFFERENT $f"; fi; done; ls ../new | sort > /tmp/n.$$; ls | sort | diff - /tmp/n.$$ && echo "same file list") | tee $OUT/${TAG}_dump_compare.txt
rm -rf $DUMP /tmp/n.$$
fi
if [ $STAGE = tests ]; then
[ -f $OUT/${TAG}_smoke.log ] || { timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${TAG}_smoke.log 2>&1; echo "smoke exit $?"; tail -n 2 $OUT/${TAG}_smoke.log; }
FILES=("${@:5}"); [ ${#FILES[@]} -eq 0 ] && FILES=(tests)
timeout 1800 python -m pytest "${FILES[@]}" -q -m gpu > $OUT/${TAG}_pytest_gpu_$(basename ${5:-all} .py).log 2>&1; echo "pytest gpu exit $?"; tail -n 3 $OUT/${TAG}_pytest_gpu_$(basename ${5:-all} .py).log
fi
