#!/bin/bash
# round 4: k-way replay batch phase -- its GPU tests, then parent/new A/B of the bench value (3 processes each, alternated),
# byte comparison of --dump-outputs, the phase split (-DQA_RP_PROFILE builds) of both; then the whole GPU suite and smoke()
# on the k-way build, one full bench line, and configs 2 and 4 on parent and new builds.  The parent half of this call failed
# (the new Python layer binds qa_model_replay_kway, which the parent library lacks); gpu_r4d.sh redoes it from a parent checkout
set -u
o=${1:?usage: $0 OUTPUT_DIR}
P=$PWD/build/variants/parent.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $o/r4b_gpu.txt 2>&1
timeout 900 python -m pytest tests/test_gpu_replay_kway.py -q -x > $o/r4b_kway_tests.log 2>&1
rc=$?
tail -3 $o/r4b_kway_tests.log
if [ $rc -ne 0 ]; then exit $rc; fi
B="python bench.py --gpus 1 --steps 3 --warmup 3 --no-full-job --no-e2e --no-cpu-baseline"
: > $o/r4b_ab.log
for i in 1 2 3; do
  for v in parent new; do
    d=""; if [ $i = 1 ]; then d="--dump-outputs $o/r4b_dump_$v"; fi
    if [ $v = parent ]; then QA_LIB_PATH=$P timeout 400 $B $d > $o/r4b_bench_${v}_$i.json 2>> $o/r4b_ab.log
    else timeout 400 $B $d > $o/r4b_bench_${v}_$i.json 2>> $o/r4b_ab.log; fi
    echo "$v $i $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print(d['value'])" $o/r4b_bench_${v}_$i.json)" >> $o/r4b_ab.log
  done
done
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv >> $o/r4b_gpu.txt 2>&1
(cd $o && sha256sum r4b_dump_parent/* r4b_dump_new/*) > $o/r4b_dump_sha.txt
rm -rf $o/r4b_dump_parent $o/r4b_dump_new
QA_LIB_PATH=$PWD/build/variants/parent_prof.so timeout 300 python tools/probe_replay.py --sweeps 50 > $o/r4b_split_parent.log 2>&1
grep -v "qa sweep" $o/r4b_split_parent.log > $o/r4b_split_parent_summary.log
QA_LIB_PATH=$PWD/build/variants/kway_prof.so timeout 300 python tools/probe_replay.py --sweeps 50 > $o/r4b_split_new.log 2>&1
grep -v "qa sweep" $o/r4b_split_new.log > $o/r4b_split_new_summary.log
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $o/r4c_gpu.txt 2>&1
timeout 1500 python -m pytest tests -q -m gpu > $o/r4c_tests.log 2>&1
echo "tests rc=$?" >> $o/r4c_tests.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $o/r4c_smoke.log 2>&1
timeout 900 python bench.py --gpus 1 --steps 3 --warmup 3 > $o/r4c_bench_full.json 2> $o/r4c_bench_full.err
for v in parent new; do
  if [ $v = parent ]; then L=$P; else L=$PWD/scrna_seq_qannealing_clustering_b200/csrc/libqanneal.so; fi
  QA_LIB_PATH=$L timeout 300 python tools/probe_c2.py > $o/r4c_c2_$v.log 2>&1
  QA_LIB_PATH=$L timeout 400 python tools/probe_c4.py > $o/r4c_c4_$v.log 2>&1
done
cat $o/r4b_ab.log | grep -v '^\[' | tail -6; tail -2 $o/r4c_tests.log; tail -1 $o/r4c_smoke.log
