"""PopulationEvaluator against a loop of P Evaluator.evaluate calls at n envs each (default options, features-only
stepping, one episode per env, greedy). Prints one JSON line (and writes it to --out).

Per (P, n): the wall time of one evaluate call (host clock around it: it ends by copying the results to the host) for the
population evaluator and for the loop of P calls on one Evaluator(n), median of --repeats after --warmup, and the
env-steps/s of each (P n max_turns per call). The kernel time per row of wab_policy_act_population against
wab_policy_forward_population on the same P n rows (CUDA events around --launches launches of each, alternating, median
of --repeats). At --pbt (P x n) the time of one PBT ready event (evaluation, ranking, exploit, explore) beside one
PPOPopulation iteration. The GPU's name, power limit and max SM clock are read in the same run."""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.bench_train import gpu_info  # noqa: E402


def _policies(P, flat_dim, n_actions):
    from wab_gym_b200.policy import Policy
    torch.manual_seed(0)
    return [Policy(flat_dim, n_actions).cuda() for _ in range(P)]


def _median_wall(fn, warmup, repeats):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    times.sort()
    return times[len(times) // 2]


def _event_time(fn, launches):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(launches):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / 1e3 / launches


def eval_arms(P, n, warmup, repeats, launches):
    from wab_gym_b200 import Evaluator, PopulationEvaluator
    pe = PopulationEvaluator(P, n, seed=1)
    pols = _policies(P, pe.flat_dim, pe.n_actions)
    t_pop = _median_wall(lambda: pe.evaluate(pols), warmup, repeats)
    # the two population forwards on the evaluator's own rows (the start state's features)
    pe.restore(pols)
    tc, f, a = pe._tc, pe.env.last_features, pe._actions
    act = lambda: tc._launch(None, f, a, None, None, None, None, 0.01, pe._ctr, 0.01)
    smp = lambda: tc._launch(pe.sample_seed, f, a, None, None, None, None, 0.01, pe._ctr, 0.01)
    for fn in (act, smp):
        _event_time(fn, 10)
    ta, ts = [], []
    for _ in range(repeats):
        ta.append(_event_time(act, launches))
        ts.append(_event_time(smp, launches))
    ta.sort(); ts.sort()
    steps = P * n * pe.steps
    pe.close()
    ev = Evaluator(n, seed=1)
    t_loop = _median_wall(lambda: [ev.evaluate(p) for p in pols], warmup, repeats)
    ev.close()
    torch.cuda.empty_cache()
    return {"members": P, "envs_per_member": n, "total_envs": P * n, "env_steps_per_call": steps,
            "population": {"call_s": t_pop, "env_steps_per_s": steps / t_pop},
            "evaluator_loop": {"call_s": t_loop, "env_steps_per_s": steps / t_loop},
            "speedup": t_loop / t_pop,
            "kernel_ns_per_row": {"act_population": ta[len(ta) // 2] / (P * n) * 1e9,
                                  "forward_population": ts[len(ts) // 2] / (P * n) * 1e9}}


def pbt_arm(P, n, warmup, repeats):
    from wab_gym_b200 import PopulationBasedTraining, PopulationEvaluator, PPOPopulation, VecEnv
    env = VecEnv(P * n, seed=1, features=True, emit_grids=False)
    pols = _policies(P, env.flat_dim, env.n_actions)
    pop = PPOPopulation(env, P, policies=pols)
    pbt = PopulationBasedTraining(pop, PopulationEvaluator(P, n, seed=2), fraction=0.25)
    it = _median_wall(pop.train_iteration, warmup, repeats)
    ready = _median_wall(pbt.ready, 1, repeats)
    evaluate = _median_wall(lambda: pbt.evaluator.evaluate(pop.policies), 1, repeats)
    env.close()
    return {"members": P, "envs_per_member": n, "horizon": pop.horizon, "iteration_s": it, "ready_event_s": ready,
            "of_which_evaluate_s": evaluate}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="1x32768,4x8192,16x2048,64x512", help="comma-separated P x n")
    ap.add_argument("--pbt", default="16x2048", help="P x n of the ready-event measurement ('' to skip)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_population_eval.py measures on a CUDA device; there is none here")
    res = {"bench": "population_eval", "episodes_per_env": 1, "greedy": True, "stepping": "features-only",
           "options": "default", **gpu_info(), "results": []}
    for cfg in a.configs.split(","):
        P, n = (int(x) for x in cfg.split("x"))
        entry = eval_arms(P, n, a.warmup, a.repeats, a.launches)
        res["results"].append(entry)
        print(json.dumps(entry), file=sys.stderr, flush=True)
    if a.pbt:
        P, n = (int(x) for x in a.pbt.split("x"))
        res["pbt"] = pbt_arm(P, n, a.warmup, a.repeats)
        print(json.dumps(res["pbt"]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
