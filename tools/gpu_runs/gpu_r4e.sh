#!/bin/bash
# round 4, after the kernel split (k_anneal_replay<G, S, KWAY>): the k-way and replay GPU tests, smoke(), config 4 (no k-way
# blocks: the parent's kernel) and config 2 on both builds, and the bench value of both builds alternated, 2 processes each.
# The parent runs from a checkout of the parent commit (build/parent_tree) with its library in build/variants/parent.so.
set -u
o=$(cd "${1:?usage: $0 OUTPUT_DIR}" && pwd)
R=$PWD
T=$PWD/build/parent_tree
P=$R/build/variants/parent.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $o/r4e_gpu.txt 2>&1
timeout 600 python -m pytest tests/test_gpu_replay_kway.py tests/test_gpu_replay.py tests/test_gpu_interval_groups.py -q > $o/r4e_tests.log 2>&1
echo "tests rc=$?" >> $o/r4e_tests.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $o/r4e_smoke.log 2>&1
for v in parent new; do
  if [ $v = parent ]; then
    (cd $T && QA_LIB_PATH=$P timeout 400 python tools/probe_c4.py > $o/r4e_c4_$v.log 2>&1)
    (cd $T && QA_LIB_PATH=$P timeout 300 python tools/probe_c2.py > $o/r4e_c2_$v.log 2>&1)
  else
    timeout 400 python tools/probe_c4.py > $o/r4e_c4_$v.log 2>&1
    timeout 300 python tools/probe_c2.py > $o/r4e_c2_$v.log 2>&1
  fi
done
B="python bench.py --gpus 1 --steps 3 --warmup 3 --no-full-job --no-e2e --no-cpu-baseline"
: > $o/r4e_ab.log
for i in 1 2; do
  for v in parent new; do
    d=""; if [ $i = 1 ]; then d="--dump-outputs $o/r4e_dump_$v"; fi
    if [ $v = parent ]; then (cd $T && QA_LIB_PATH=$P timeout 400 $B $d > $o/r4e_bench_${v}_$i.json 2>> $o/r4e_ab.err)
    else timeout 400 $B $d > $o/r4e_bench_${v}_$i.json 2>> $o/r4e_ab.err; fi
    echo "$v $i $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print(d['value'], d['ms_per_step'], d['clocks']['sm_mhz'], d['config5']['value'])" $o/r4e_bench_${v}_$i.json)" >> $o/r4e_ab.log
  done
done
(cd $o && sha256sum r4e_dump_parent/* r4e_dump_new/*) > $o/r4e_dump_sha.txt
rm -rf $o/r4e_dump_parent $o/r4e_dump_new
tail -2 $o/r4e_tests.log; tail -1 $o/r4e_smoke.log; cat $o/r4e_ab.log; tail -1 $o/r4e_c4_parent.log $o/r4e_c4_new.log
