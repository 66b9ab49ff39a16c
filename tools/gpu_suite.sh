#!/bin/bash
# Run the GPU parity suite file by file under a timeout (a hung kernel must not take the box down).
# usage: tools/gpu_suite.sh [pytest -k expression]
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,driver_version,memory.total,clocks.max.sm --format=csv > gpurun_out/gpu_info.txt 2>&1
status=0
for path in tests/test_gpu_*.py; do
  f=$(basename "$path" .py)
  timeout -k 10 900 python -m pytest "$path" -q -m gpu --maxfail=12 --no-header -p no:cacheprovider ${1:+-k "$1"} \
      > gpurun_out/$f.log 2>&1
  rc=$?
  echo "== $f exit $rc"
  tail -n 25 gpurun_out/$f.log
  [ $rc -ne 0 ] && status=1
done
exit $status
