#!/bin/sh
# A/B of two builds of the library on the same box: tools/ab.sh <libA> <libB> [sizes...]
. "$(dirname "$0")/window_steps.sh"
A=$1; B=$2; shift 2
for n in "$@"; do
  for rep in 1 2; do
    for lib in $A $B; do
      WAB_LIB=$lib python bench.py --num-envs $n --steps "$(window_steps $n)" --warmup 16 --skip-e2e --skip-cpu 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('$lib', $n, '%.4g' % d['value'], 'per_call %.4g' % d['per_call']['value'], d['clocks']['sm_mhz'])"
    done
  done
done
