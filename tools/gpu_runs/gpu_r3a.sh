#!/bin/bash
# k_energy: load batches of 8 / 16 / 32 couplers (A/B), energy tests on the new default
set -u
o=gpurun_out
: > $o/r3b_energy.log
for v in base; do
  echo "== $v" >> $o/r3b_energy.log
  if [ $v = base ]; then timeout 120 python tools/probe_energy.py >> $o/r3b_energy.log 2>&1
  else QA_LIB_PATH=$PWD/build/variants/$v.so timeout 120 python tools/probe_energy.py >> $o/r3b_energy.log 2>&1; fi
done
timeout 200 python -m pytest tests/test_gpu_parity.py tests/test_gpu_fullsize.py -q -m gpu > $o/r3b_tests.log 2>&1
