#!/bin/bash
# Same-box A/B of the two-warp pipeline kernel (WAB_PIPE) across lanes-per-env variants and batch sizes. Developer tool.
cd "$(dirname "$0")/.."
. tools/window_steps.sh
for n in ${SIZES:-4096}; do
 for lpe in ${LPES:-4 8 16}; do
  for pipe in 0 1; do
    WAB_LPE=$lpe WAB_PIPE=$pipe python bench.py --num-envs $n --steps "$(window_steps $n)" --warmup 5 --legs none --skip-e2e --skip-cpu --leg-window-ms 50 | python -c "
import json,sys
d=json.loads(sys.stdin.read())
print('n $n lpe $lpe pipe $pipe', d['roofline']['kernel'], 'value %.4g'%d['value'], 'per_call %.4g'%d['per_call']['value'])"
  done
 done
done
