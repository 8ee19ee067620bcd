#!/bin/bash
# round 4, A/B again: the parent runs from a checkout of the parent commit (build/parent_tree, its library built into
# build/variants/parent.so), since the new Python layer binds a C function the parent library does not have.  3 processes of
# each build alternated, --dump-outputs byte comparison, phase split of both builds, configs 2 and 4 on both.
set -u
o=$(cd "${1:?usage: $0 OUTPUT_DIR}" && pwd)
R=$PWD
T=$PWD/build/parent_tree
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $o/r4d_gpu.txt 2>&1
B="python bench.py --gpus 1 --steps 3 --warmup 3 --no-full-job --no-e2e --no-cpu-baseline"
: > $o/r4d_ab.log
for i in 1 2 3; do
  for v in parent new; do
    d=""; if [ $i = 1 ]; then d="--dump-outputs $o/r4d_dump_$v"; fi
    if [ $v = parent ]; then (cd $T && QA_LIB_PATH=$R/build/variants/parent.so timeout 400 $B $d > $o/r4d_bench_${v}_$i.json 2>> $o/r4d_ab.err)
    else timeout 400 $B $d > $o/r4d_bench_${v}_$i.json 2>> $o/r4d_ab.err; fi
    echo "$v $i $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print(d['value'], d['ms_per_step'], d['clocks']['sm_mhz'])" $o/r4d_bench_${v}_$i.json)" >> $o/r4d_ab.log
  done
done
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv >> $o/r4d_gpu.txt 2>&1
(cd $o && sha256sum r4d_dump_parent/* r4d_dump_new/*) > $o/r4d_dump_sha.txt
rm -rf $o/r4d_dump_parent $o/r4d_dump_new
(cd $T && QA_LIB_PATH=$R/build/variants/parent_prof.so timeout 300 python tools/probe_replay.py --sweeps 50 > $o/r4d_split_parent.log 2>&1)
grep -v "qa sweep" $o/r4d_split_parent.log > $o/r4d_split_parent_summary.log
for v in parent new; do
  if [ $v = parent ]; then
    (cd $T && QA_LIB_PATH=$R/build/variants/parent.so timeout 300 python tools/probe_c2.py > $o/r4d_c2_$v.log 2>&1)
    (cd $T && QA_LIB_PATH=$R/build/variants/parent.so timeout 400 python tools/probe_c4.py > $o/r4d_c4_$v.log 2>&1)
  else
    timeout 300 python tools/probe_c2.py > $o/r4d_c2_$v.log 2>&1
    timeout 400 python tools/probe_c4.py > $o/r4d_c4_$v.log 2>&1
  fi
done
cat $o/r4d_ab.log; cat $o/r4d_dump_sha.txt; tail -1 $o/r4d_split_parent_summary.log
