#!/bin/bash
# A/B of build variants on the GPU box: tools/ab_variant.sh "<name>:<nvcc -D flags>" ... ; prints value / per_call at 4,096 envs
# (and at the sizes in $SIZES). Developer tool.
set -e
cd "$(dirname "$0")/.."
. tools/window_steps.sh
mkdir -p gpurun_out/variants
for spec in "$@"; do
  name="${spec%%:*}"; flags="${spec#*:}"
  lib=gpurun_out/variants/libwab_$name.so
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC -shared $flags -o $lib wab_gym_b200/csrc/wab_kernels.cu
  for n in ${SIZES:-4096}; do
    WAB_LIB=$lib python bench.py --num-envs $n --steps "$(window_steps $n)" --warmup 5 --legs none --skip-e2e --skip-cpu --leg-window-ms 50 ${BENCH_ARGS} | python -c "
import json,sys
d=json.loads(sys.stdin.read())
print('$name', $n, d['roofline']['kernel'], 'value %.4g'%d['value'], 'per_call %.4g'%d['per_call']['value'])"
  done
done
