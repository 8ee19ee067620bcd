#!/bin/bash
# round 7, dwave-samplers sample options (random variable order, Gibbs acceptance; every pre-existing kernel's SASS identical
# to the parent's: profiles/r7_sass_kernels_vs_parent.log).
# tests: the whole GPU suite and smoke() on this build.  probe: tools/probe_proposals.py.  bench: bench.py alternated between the
# parent checkout (build/parent_tree, library build/variants/parent.so) and this build; the --dump-outputs of the first
# process of each go to a temporary directory and only their hashes are kept.
# Run from the repository root on a B200, one mode per process, writing into an existing OUTPUT_DIR:
#   bash tools/gpu_runs/gpu_r7a.sh OUTPUT_DIR tests
#   bash tools/gpu_runs/gpu_r7a.sh OUTPUT_DIR probe
#   bash tools/gpu_runs/gpu_r7a.sh OUTPUT_DIR bench
#   bash tools/gpu_runs/gpu_r7a.sh OUTPUT_DIR bench-reversed
set -u
o=$(cd "${1:?usage: $0 OUTPUT_DIR tests|probe|bench|bench-reversed}" && pwd)
what=${2:?usage: $0 OUTPUT_DIR tests|probe|bench|bench-reversed}
R=$PWD
T=$PWD/build/parent_tree
P=$R/build/variants/parent.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $o/r7a_gpu_$what.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $o/r7a_build_$what.log 2>&1
echo "build rc=$?" >> $o/r7a_build_$what.log
if [ $what = tests ]; then
  timeout 1200 python -m pytest -m gpu tests -q -rfs --tb=short -p no:cacheprovider --durations=30 2>&1 | tail -c 400000 > $o/r7a_tests.log
  timeout 120 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -c 20000 > $o/r7a_smoke.log
  tail -4 $o/r7a_tests.log; tail -1 $o/r7a_smoke.log
  exit 0
fi
if [ $what = probe ]; then
  timeout 600 python tools/probe_proposals.py --out $o/r7a_probe_proposals.jsonl > /dev/null 2> $o/r7a_probe.err
  cat $o/r7a_probe_proposals.jsonl; tail -5 $o/r7a_probe.err
  exit 0
fi
if [ $what = bench-reversed ]; then   # two more pairs, this build first, flagship measurement only
  B="python bench.py --gpus 1 --steps 3 --warmup 3 --no-full-job --no-config5 --no-cpu-baseline"
  : > $o/r7a_ab_reversed.log
  for i in 1 2; do
    for v in new parent; do
      if [ $v = parent ]; then (cd $T && QA_LIB_PATH=$P timeout 400 $B > $o/r7a_rev_${v}_$i.json 2>> $o/r7a_ab.err)
      else timeout 400 $B > $o/r7a_rev_${v}_$i.json 2>> $o/r7a_ab.err; fi
      echo "$v $i $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print(d['value'], d['roofline']['ms_per_launch'], d['clocks']['sm_mhz'])" $o/r7a_rev_${v}_$i.json 2>&1 | tail -1)" >> $o/r7a_ab_reversed.log
    done
  done
  tail -c 4000 $o/r7a_ab.err > $o/r7a_ab_reversed.err.tail; rm -f $o/r7a_ab.err
  cat $o/r7a_ab_reversed.log
  exit 0
fi
D=$(mktemp -d)
B="python bench.py --gpus 1 --steps 3 --warmup 3 --no-full-job"
: > $o/r7a_ab.log
for i in 1 2; do
  for v in parent new; do
    d="--no-cpu-baseline"; if [ $i = 1 ]; then d="--dump-outputs $D/$v"; fi   # first process: dump and CPU parity
    if [ $v = parent ]; then (cd $T && QA_LIB_PATH=$P timeout 400 $B $d > $o/r7a_bench_${v}_$i.json 2>> $o/r7a_ab.err)
    else timeout 400 $B $d > $o/r7a_bench_${v}_$i.json 2>> $o/r7a_ab.err; fi
    echo "$v $i $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); p=(d.get('cpu_baseline') or {}).get('parity_check') or {}; print(d['value'], d['e2e_best_k']['value'], d['clocks']['sm_mhz'], p.get('final_states_identical_to_gpu'), p.get('energies_bitwise_identical_to_gpu'))" $o/r7a_bench_${v}_$i.json 2>&1 | tail -1)" >> $o/r7a_ab.log
  done
done
(cd $D && sha256sum parent/* new/*) > $o/r7a_dump_sha.txt
rm -rf $D
tail -c 4000 $o/r7a_ab.err > $o/r7a_ab.err.tail; rm -f $o/r7a_ab.err
cat $o/r7a_ab.log $o/r7a_dump_sha.txt
