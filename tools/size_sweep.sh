#!/bin/sh
# fused step_many throughput per batch size with the library's own choices (lanes per env, CTAs per SM)
. "$(dirname "$0")/window_steps.sh"
for n in "$@"; do
  python bench.py --num-envs $n --steps "$(window_steps $n)" --warmup 16 --skip-e2e --skip-cpu 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('n $n value %.4g per_call %.4g frac %.3f' % (d['value'], d['per_call']['value'], d['roofline']['frac']))"
done
