"""PPOPopulation against a loop of P standalone PPOTrainers at equal total envs (default 32,768 = P n; default options,
features-only stepping, horizon 64, 4 epochs x 4 minibatches). Prints one JSON line (and writes it to --out).

Per (P, n): the iteration time of the population and of the loop that runs one train_iteration of each of the P trainers,
each on its own VecEnv(n, env_id_base=p n) (CUDA events around the iteration, median of --repeats after --warmup), the
collected env-steps/s (P n horizon per iteration), torch.cuda.max_memory_allocated over the timed iterations, and the
PPO backward of one minibatch: one wab_policy_ppo_backward_population launch against the P wab_policy_ppo_backward
launches of the loop (CUDA events around all of them, median of --repeats). The GPU's name, power limit and max SM clock
are read in the same run."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.bench_train import gpu_info  # noqa: E402


def _median_time(fn, warmup, repeats):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(repeats):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e) / 1e3)
    times.sort()
    return times[len(times) // 2]


def population_arm(P, n, horizon, warmup, repeats):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.population import PPOPopulation
    env = VecEnv(P * n, seed=1, features=True, emit_grids=False)
    torch.manual_seed(0)
    pop = PPOPopulation(env, P, policies=[Policy(env.flat_dim, env.n_actions) for _ in range(P)], horizon=horizon)
    for _ in range(warmup):
        pop.train_iteration()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    it = _median_time(pop.train_iteration, 0, repeats)
    peak = torch.cuda.max_memory_allocated()
    b, m = pop.last_batch, pop._bounds[1]
    rows = pop._mb_rows[0]
    coefs = [(hp["clip_eps"], 1.0 / m, hp["vf_coef"] / m, hp["ent_coef"] / m) for hp in pop.hyperparameters]
    bwd = _median_time(lambda: pop._tc.ppo_backward(b["features"], b["counters"], b["actions"], b["logp"], b["advantage"],
                                                    b["target"], rows, pop._mb_counts[0], coefs, out=pop._grad,
                                                    logp=pop._new["logp"], value=pop._new["value"],
                                                    entropy=pop._new["entropy"]), 3, repeats)
    del pop
    env.close()
    torch.cuda.empty_cache()
    return it, peak, bwd


def loop_arm(P, n, horizon, warmup, repeats):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    trs = []
    torch.manual_seed(0)
    for p in range(P):
        env = VecEnv(n, seed=1, env_id_base=p * n, features=True, emit_grids=False)
        trs.append(PPOTrainer(env, Policy(env.flat_dim, env.n_actions), horizon=horizon))

    def iteration():
        for tr in trs:
            tr.train_iteration()
    for _ in range(warmup):
        iteration()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    it = _median_time(iteration, 0, repeats)
    peak = torch.cuda.max_memory_allocated()
    args = []
    for tr in trs:
        b, m = tr.last_batch, float(tr._bounds[1])
        args.append(((b["features"], b["counters"], b["actions"], b["logp"], b["advantage"], b["target"],
                      tr._perm[:tr._bounds[1]], tr._counts[:1], tr.clip_eps, 1.0 / m, tr.vf_coef / m, tr.ent_coef / m),
                     dict(out=tr._grad, logp=tr._new["logp"], value=tr._new["value"], entropy=tr._new["entropy"])))

    def backward():
        for tr, (a, kw) in zip(trs, args):
            tr._tc.ppo_backward(*a, **kw)
    bwd = _median_time(backward, 3, repeats)
    for tr in trs:
        tr.env.close()
    del trs, args
    torch.cuda.empty_cache()
    return it, peak, bwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="1x32768,4x8192,16x2048,64x512", help="comma-separated P x n")
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_population.py measures on a CUDA device; there is none here")
    res = {"bench": "population", "horizon": a.horizon, "epochs": 4, "minibatches": 4, "stepping": "features-only",
           "options": "default", **gpu_info(), "results": []}
    for cfg in a.configs.split(","):
        P, n = (int(x) for x in cfg.split("x"))
        steps = P * n * a.horizon
        pit, ppeak, pbwd = population_arm(P, n, a.horizon, a.warmup, a.repeats)
        lit, lpeak, lbwd = loop_arm(P, n, a.horizon, a.warmup, a.repeats)
        entry = {"members": P, "envs_per_member": n, "total_envs": P * n,
                 "population": {"iteration_s": pit, "env_steps_per_s": steps / pit, "backward_minibatch_s": pbwd,
                                "peak_alloc_bytes": ppeak},
                 "standalone_loop": {"iteration_s": lit, "env_steps_per_s": steps / lit, "backward_minibatch_s": lbwd,
                                     "peak_alloc_bytes": lpeak},
                 "speedup_iteration": lit / pit, "speedup_backward": lbwd / pbwd}
        res["results"].append(entry)
        print(json.dumps(entry), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
