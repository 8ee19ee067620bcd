#!/bin/bash
# round 5, output-stage tests.  tests: the new output-stage tests against the parent's library (which of them fail before the
# fix; tests-new leaves that part out), then the whole GPU suite and smoke() on this build.  bench: bench.py alternated between the parent checkout
# (build/parent_tree, library build/variants/parent.so) and this build; the --dump-outputs of the first process of each go to
# a temporary directory and only their hashes are kept.
set -u
o=$(cd "${1:?usage: $0 OUTPUT_DIR tests|tests-new|bench}" && pwd)
what=${2:?usage: $0 OUTPUT_DIR tests|tests-new|bench}
R=$PWD
T=$PWD/build/parent_tree
P=$R/build/variants/parent.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $o/r5a_gpu_$what.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $o/r5a_build_$what.log 2>&1
echo "build rc=$?" >> $o/r5a_build_$what.log
if [ $what = tests ] || [ $what = tests-new ]; then
  [ $what = tests ] && QA_LIB_PATH=$P timeout 300 python -m pytest -m gpu tests/test_gpu_output_stage.py "tests/test_gpu_interval_groups.py::test_max_groups_wide_coefficients" \
    -q -rf --tb=line -p no:cacheprovider 2>&1 | tail -c 200000 > $o/r5a_parent_tests.log
  timeout 780 python -m pytest -m gpu tests -q -rfs --tb=short -p no:cacheprovider --durations=30 2>&1 | tail -c 400000 > $o/r5a_tests.log
  timeout 120 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -c 20000 > $o/r5a_smoke.log
  [ $what = tests ] && tail -4 $o/r5a_parent_tests.log; tail -4 $o/r5a_tests.log; tail -1 $o/r5a_smoke.log
  exit 0
fi
D=$(mktemp -d)
B="python bench.py --gpus 1 --steps 3 --warmup 3 --no-full-job"
: > $o/r5a_ab.log
for i in 1 2; do
  for v in parent new; do
    d="--no-cpu-baseline"; if [ $i = 1 ]; then d="--dump-outputs $D/$v"; fi   # first process: dump and CPU parity
    if [ $v = parent ]; then (cd $T && QA_LIB_PATH=$P timeout 400 $B $d > $o/r5a_bench_${v}_$i.json 2>> $o/r5a_ab.err)
    else timeout 400 $B $d > $o/r5a_bench_${v}_$i.json 2>> $o/r5a_ab.err; fi
    echo "$v $i $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); p=(d.get('cpu_baseline') or {}).get('parity_check') or {}; print(d['value'], d['e2e_best_k']['value'], d['clocks']['sm_mhz'], p.get('final_states_identical_to_gpu'), p.get('energies_bitwise_identical_to_gpu'))" $o/r5a_bench_${v}_$i.json 2>&1 | tail -1)" >> $o/r5a_ab.log
  done
done
(cd $D && sha256sum parent/* new/*) > $o/r5a_dump_sha.txt
rm -rf $D
tail -c 4000 $o/r5a_ab.err > $o/r5a_ab.err.tail; rm -f $o/r5a_ab.err
cat $o/r5a_ab.log $o/r5a_dump_sha.txt
