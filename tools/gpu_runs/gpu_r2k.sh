#!/bin/bash
# round-2: full GPU suite on the split library, dense-kernel variants, ncu sections of the benched replay launch (hardware-counter
# sections only: instrumented sections change the shared-memory base and slow a 7 s persistent kernel beyond reason)
set -u
o=gpurun_out
timeout 900 python -m pytest tests -q -m gpu -x > $o/r2k_tests.log 2>&1
: > $o/r2k_ab_dense.log
for v in base dn_lop3 dn_c3 dn_lop3_c3; do
  for reads in 37888 56832; do
    echo "== $v reads $reads" >> $o/r2k_ab_dense.log
    if [ $v = base ]; then timeout 300 python tools/probe_c5.py --reads $((reads/2)) --ref-reads 0 2>&1 | grep -E "reads $reads |Error|error" >> $o/r2k_ab_dense.log
    else QA_LIB_PATH=$PWD/build/variants/$v.so timeout 300 python tools/probe_c5.py --reads $((reads/2)) --ref-reads 0 2>&1 | grep -E "reads $reads |Error|error" >> $o/r2k_ab_dense.log; fi
  done
done
timeout 420 ncu --replay-mode application --section SpeedOfLight --section WarpStateStats --section SchedulerStats --section Occupancy \
   --section LaunchStats --clock-control none -k regex:k_anneal_replay -c 1 \
   -o $o/r2k_replay_sections -f python tools/profile_run.py --workload c3 --reads 75776 --sweeps 50 > $o/r2k_ncu_replay.log 2>&1
ls -la $o/*.ncu-rep >> $o/r2k_ncu_replay.log 2>&1
