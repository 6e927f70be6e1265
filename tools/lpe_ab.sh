#!/bin/sh
# lanes-per-env sweep at the given batch sizes (fused step_many, 256 steps per launch)
. "$(dirname "$0")/window_steps.sh"
for n in "$@"; do for lpe in 1 4 8 16 32; do
  WAB_LPE=$lpe python bench.py --num-envs $n --steps "$(window_steps $n)" --warmup 16 --skip-e2e --skip-cpu 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('n $n lpe $lpe value %.4g per_call %.4g' % (d['value'], d['per_call']['value']))"
done; done
