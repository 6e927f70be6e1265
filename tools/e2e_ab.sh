#!/bin/sh
# e2e (host buffers) A/B: staged copies (0) vs the thread-per-env kernel writing the pinned host block directly (1)
for n in "$@"; do
for m in 0 1; do
  WAB_HOST_MAPPED=$m python bench.py --num-envs $n --steps 256 --warmup 8 --skip-cpu 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('n $n mapped $m e2e %.4g  us/step %.2f' % (d['e2e']['value'], d['e2e']['ms_per_step']*1e3))"
done; done
