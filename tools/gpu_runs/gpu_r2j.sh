#!/bin/bash
# round-2: dense-kernel build variants A/B, recursion tests (all rules), ncu captures of the benched replay launch (sections,
# application replay) and of the dense kernel (full set)
set -u
o=gpurun_out
timeout 600 python -m pytest tests/test_gpu_recursion.py -q -m gpu > $o/r2j_rec_tests.log 2>&1
: > $o/r2j_ab_dense.log
for v in base dn_lop3 dn_c3 dn_lop3_c3; do
  for reads in 37888 56832; do
    echo "== $v reads $reads" >> $o/r2j_ab_dense.log
    if [ $v = base ]; then timeout 300 python tools/probe_c5.py --reads $((reads/2)) --ref-reads 0 2>&1 | grep "reads $reads " >> $o/r2j_ab_dense.log
    else QA_LIB_PATH=$PWD/build/variants/$v.so timeout 300 python tools/probe_c5.py --reads $((reads/2)) --ref-reads 0 2>&1 | grep "reads $reads " >> $o/r2j_ab_dense.log; fi
  done
done
# dense kernel: plain run, then the full ncu set on one launch (small read count: the per-SM shape is the same, 8 warps per SM)
timeout 300 python tools/profile_run.py --workload c5 --reads 37888 --sweeps 2 > $o/r2j_c5_plain.log 2>&1 && \
timeout 900 ncu --set full --import-source on --clock-control none -k regex:k_anneal_dense -c 1 -o $o/r2j_dense_full -f \
   python tools/profile_run.py --workload c5 --reads 37888 --sweeps 2 > $o/r2j_ncu_dense.log 2>&1
# replay kernel at the benched launch shape: plain run, then sections by application replay (kernel replay would save / restore ~100 GB per pass)
timeout 300 python tools/profile_run.py --workload c3 --reads 75776 --sweeps 50 > $o/r2j_c3_plain.log 2>&1 && \
timeout 1200 ncu --replay-mode application --section SpeedOfLight --section WarpStateStats --section SchedulerStats --section Occupancy \
   --section LaunchStats --section MemoryWorkloadAnalysis --section InstructionStats --clock-control none -k regex:k_anneal_replay -c 1 \
   -o $o/r2j_replay_sections -f python tools/profile_run.py --workload c3 --reads 75776 --sweeps 50 > $o/r2j_ncu_replay.log 2>&1
ls -la $o/*.ncu-rep >> $o/r2j_ncu_replay.log 2>&1
