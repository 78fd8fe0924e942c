#!/bin/bash
# Tuning helper: build variant libraries of the same sources with -D flags (no GPU needed, through
# decombinator_b200/build.py, so that they are compiled and linked exactly as libdcb.so is) and bench each on a GPU.
#   tools/variants.sh build  NAME "-DFLAG=1 ..." [NAME2 "..."]...     -> build/libdcb_var_NAME.so
#   tools/variants.sh bench  [extra bench.py args]                      -> build/variants.txt
set -e
cd "$(dirname "$0")/.."
if [ "$1" == "build" ]; then
  shift; pids=()
  while [ $# -ge 2 ]; do
    python -m decombinator_b200.build --variant "var_$1" $2 &
    pids+=($!)
    shift 2
  done
  for p in "${pids[@]}"; do wait "$p"; done
  ls -la build/
else
  shift || true
  mkdir -p build; : > build/variants.txt
  for f in build/libdcb_var_*.so; do
    for rep in 1 2; do
      DCB_LIB=$PWD/$f timeout 300 python bench.py --steps 20 --warmup 3 --no-cpu-baseline "$@" 2>/dev/null | python -c "
import sys,json
d=json.loads(sys.stdin.readline()); print('$f', '%.2f G reads/s  exact %.4f ms  general %.3f ms  e2e %.3f G' % (d['value']/1e9, d['kernels_ms']['dcb_exact_kernel'], d['kernels_ms']['dcb_general_kernel'], d['e2e']['value']/1e9))" >> build/variants.txt || echo "$f FAILED" >> build/variants.txt
    done
  done
  cat build/variants.txt
fi
