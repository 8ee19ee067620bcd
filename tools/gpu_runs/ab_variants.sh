#!/bin/bash
# development aid: A/B of kernel build variants (build/variants/*.so from tools/build_variant.py, built with extra -D flags) on the bench workload
set -u
out=gpurun_out/$1; shift
: > $out
run() { # name lib args...
  local name=$1 lib=$2; shift 2
  echo "== $name ($lib) $*" >> $out
  if [ "$lib" = base ]; then timeout 600 python tools/probe_replay.py "$@" >> $out 2>&1
  else QA_LIB_PATH=$PWD/build/variants/$lib.so timeout 600 python tools/probe_replay.py "$@" >> $out 2>&1; fi
}
"$@"
