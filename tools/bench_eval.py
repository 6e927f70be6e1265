"""Cost of evaluation: the greedy tail against the sampling one, and Evaluator throughput; plus what PPO training does to
the evaluated policy (reported, not asserted). Prints one JSON line (and writes it to --out).

In one process, on the GPU of the current device, with its name and power limit read alongside:
- act_vs_forward: wab_policy_act (greedy) and wab_policy_forward (sampled) on the feature bytes of a reset
  features-only VecEnv, per size; CUDA events around --launches launches, --warmup rounds first, median of --repeats,
  the two calls alternating within each round; ns per row;
- evaluator: Evaluator.evaluate (restore the start state, max_turns steps of policy + env.step, first_episodes, host
  copy) at each size, greedy and sampled, host clock around the whole call (it ends in a synchronisation), one warm-up
  call then the median of --eval-repeats; env-steps per second; and play() alone (the step loop) with CUDA events;
- learning: a PPOTrainer (fixed seeds) evaluated before training and after --iterations iterations by an Evaluator of
  its own seed (greedy and sampled, input noise on): EvalResult.summary() of each, and the per-episode paired difference
  (trained - initial) with its standard error, beside the unpaired standard error the same episode count would have."""
import argparse
import json
import math
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.bench_train import gpu_info  # noqa: E402


def event_median(fns, launches, warmup, repeats):
    """Per fn: median seconds per launch over `repeats` rounds of `launches` launches, the fns alternating."""
    for _ in range(warmup):
        for fn in fns:
            fn()
    torch.cuda.synchronize()
    times = [[] for _ in fns]
    for _ in range(repeats):
        for i, fn in enumerate(fns):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(launches):
                fn()
            e.record()
            e.synchronize()
            times[i].append(s.elapsed_time(e) / 1e3 / launches)
    return [statistics.median(t) for t in times]


def act_vs_forward(n, launches, warmup, repeats):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy, PolicyTrunkTC, stacked_heads
    env = VecEnv(n, seed=1, features=True, emit_grids=False)
    env.reset()
    torch.manual_seed(0)
    pol = Policy(env.flat_dim, env.n_actions).cuda()
    tc, heads = PolicyTrunkTC(env, pol), stacked_heads(pol)
    feats = env.last_features.clone()
    ctr = torch.ones(1, dtype=torch.int64, device="cuda")
    acts, value = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, device="cuda")
    logp = torch.empty(n, device="cuda")
    act = lambda: tc.forward_greedy(feats, heads, acts, value=value, logp=logp, counter=ctr)
    fwd = lambda: tc.forward_sample(feats, heads, acts, value=value, logp=logp, counter=ctr, seed=7)
    t_act, t_fwd = event_median([act, fwd], launches, warmup, repeats)
    env.close()
    return {"rows": n, "act_ns_per_row": t_act / n * 1e9, "forward_ns_per_row": t_fwd / n * 1e9, "act_over_forward": t_act / t_fwd}


def evaluator_rate(n, repeats):
    from wab_gym_b200 import Evaluator
    from wab_gym_b200.policy import Policy
    ev = Evaluator(n, seed=2)
    torch.manual_seed(0)
    pol = Policy(ev.flat_dim, ev.n_actions).cuda()
    out = {"envs": n, "steps": ev.steps}
    for greedy in (True, False):
        kind = "greedy" if greedy else "sampled"
        ev.evaluate(pol, greedy=greedy)                                  # warm-up
        walls = []
        for _ in range(repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev.evaluate(pol, greedy=greedy)
            walls.append(time.perf_counter() - t0)
        ev.restore(pol)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ev.play(greedy=greedy)
        e.record()
        e.synchronize()
        play_s = s.elapsed_time(e) / 1e3
        wall = statistics.median(walls)
        out[kind] = {"evaluate_s": wall, "env_steps_per_s": n * ev.steps / wall, "play_s": play_s,
                     "play_env_steps_per_s": n * ev.steps / play_s}
    ev.close()
    return out


def _paired(a, b):
    d = (b.returns - a.returns).reshape(-1).double()
    m = d.numel()
    sd_d = float(d.std()) if m > 1 else float("nan")
    unpaired = math.sqrt((float(a.returns.double().var()) + float(b.returns.double().var())) / m) if m > 1 else float("nan")
    return {"mean_diff": float(d.mean()), "paired_se": sd_d / math.sqrt(m), "unpaired_se": unpaired}


def learning(train_envs, eval_envs, iterations):
    from wab_gym_b200 import Evaluator, VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    env = VecEnv(train_envs, seed=1, features=True, emit_grids=False)
    torch.manual_seed(0)
    tr = PPOTrainer(env, Policy(env.flat_dim, env.n_actions))
    ev = Evaluator(eval_envs, seed=12345)
    before = {g: ev.evaluate(tr.policy, greedy=g) for g in (True, False)}
    t0 = time.time()
    for _ in range(iterations):
        tr.train_iteration()
    torch.cuda.synchronize()
    train_s = time.time() - t0
    after = {g: ev.evaluate(tr.policy, greedy=g) for g in (True, False)}
    out = {"train_envs": train_envs, "eval_envs": eval_envs, "iterations": iterations, "horizon": tr.horizon,
           "train_s": round(train_s, 2), "train_seed": 1, "eval_seed": 12345}
    for g, kind in ((True, "greedy"), (False, "sampled")):
        out[kind] = {"initial": before[g].summary(), "trained": after[g].summary(), "paired": _paired(before[g], after[g])}
    env.close()
    ev.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="32768,262144")
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=11)
    ap.add_argument("--eval-repeats", type=int, default=3)
    ap.add_argument("--train-envs", type=int, default=32768)
    ap.add_argument("--eval-envs", type=int, default=32768)
    ap.add_argument("--iterations", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py measures on a CUDA device; there is none here")
    sizes = [int(s) for s in a.sizes.split(",")]
    res = {"bench": "eval", **gpu_info(), "options": "default", "stepping": "features-only", "launches": a.launches,
           "warmup": a.warmup, "repeats": a.repeats, "eval_repeats": a.eval_repeats}
    res["act_vs_forward"] = []
    for n in sizes:
        res["act_vs_forward"].append(act_vs_forward(n, a.launches, a.warmup, a.repeats))
        print(json.dumps(res["act_vs_forward"][-1]), file=sys.stderr, flush=True)
    res["evaluator"] = []
    for n in sizes:
        res["evaluator"].append(evaluator_rate(n, a.eval_repeats))
        print(json.dumps(res["evaluator"][-1]), file=sys.stderr, flush=True)
        torch.cuda.empty_cache()
    if a.iterations > 0:
        res["learning"] = learning(a.train_envs, a.eval_envs, a.iterations)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
