#!/bin/bash
# A/B of two source trees on one GPU box, alternating: tools/ab_trees.sh <treeA> <treeB> [repetitions]. Each tree runs
# from its own directory with its own library: bench.py's headline and its 131,072 / 1,048,576-env legs, a PPOTrainer
# iteration at 32,768 envs and a PPOPopulation iteration at 16 x 2,048 (tools/bench_population.py's population arm).
# Prints one line per (repetition, tree A or B, measurement). Developer tool.
set -e
A=$(cd "$1" && pwd); B=$(cd "$2" && pwd); REPS=${3:-3}
for rep in $(seq 1 "$REPS"); do
  for tree in "$A" "$B"; do
    cd "$tree"
    label=$([ "$tree" = "$A" ] && echo A || echo B)
    python bench.py --gpus 1 --steps 131072 --warmup 64 --legs large_batch,batch_1m --skip-e2e --skip-cpu 2>/dev/null | python -c "
import json, sys
d = json.loads(sys.stdin.read().strip().splitlines()[-1])
legs = ' '.join('%s %.4g' % (k, v.get('value', float('nan'))) for k, v in d['legs'].items())
print('$label', $rep, 'bench headline %.4g per_call %.4g' % (d['value'], d['per_call']['value']), legs, 'sm_mhz', d['clocks'].get('sm_mhz'))"
    python -c "
import sys, torch
sys.path.insert(0, '.')
from tools.bench_population import population_arm, _median_time
from wab_gym_b200 import VecEnv
from wab_gym_b200.policy import Policy
from wab_gym_b200.ppo import PPOTrainer
env = VecEnv(32768, seed=1, features=True, emit_grids=False)
torch.manual_seed(0)
tr = PPOTrainer(env, Policy(env.flat_dim, env.n_actions))
t = _median_time(tr.train_iteration, 2, 5)
env.close(); del tr; torch.cuda.empty_cache()
it, _, _ = population_arm(16, 2048, 64, 2, 5)
print('$label', $rep, 'ppo_trainer_iteration_s %.5f population_16x2048_iteration_s %.5f' % (t, it))"
  done
done
