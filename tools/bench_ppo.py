"""Training throughput of PPOTrainer (wab_policy_forward collection, GAE, one wab_policy_ppo_backward launch per
minibatch, global-norm clip, Adam), features-only stepping, default options. Prints one JSON line (and writes it to --out).

Per size: training env-steps/s (env-steps collected per iteration over the whole iteration, CUDA events, after --warmup
iterations, median of --repeats), torch.cuda.max_memory_allocated over one iteration, and the PPO kernel alone on the
last batch: one minibatch (its rows, weights and outputs as the trainer passes them), CUDA events, median of --repeats,
as time per row and FLOP/s counted by tools/bench_train.py:row_flops (the fp32 network's multiply-adds, not the six
bf16 products per fp32 product the tensor cores execute).

--learn BUDGET also trains A2CTrainer(tensor_cores=True) with the reference's hyper-parameters (episodic, lr 3e-2) and
PPOTrainer with its defaults from the same initial policy for BUDGET env-steps each, and reports mean episode length
(env.stats() steps / episodes) and mean episode reward (the rewards of every collected step / episodes). Reported, not
asserted."""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.bench_train import gpu_info, row_flops  # noqa: E402


def time_iterations(tr, warmup, repeats):
    for _ in range(warmup):
        tr.train_iteration()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    times = []
    for _ in range(repeats):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        tr.train_iteration()
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e) / 1e3)
    times.sort()
    return times[len(times) // 2], torch.cuda.max_memory_allocated(), base


def time_kernel(tr, repeats):
    """One minibatch of the last batch through wab_policy_ppo_backward (the reduction included)."""
    b, dev = tr.last_batch, tr.env.device
    rows = torch.randperm(b["logp"].numel(), device=dev, dtype=torch.int32)[:tr._bounds[1]]
    m = float(rows.numel())
    args = (b["features"], b["counters"], b["actions"], b["logp"], b["advantage"], b["target"], rows, tr._counts[:1],
            tr.clip_eps, 1.0 / m, tr.vf_coef / m, tr.ent_coef / m)
    kw = dict(out=tr._grad, logp=tr._new["logp"], value=tr._new["value"], entropy=tr._new["entropy"])
    for _ in range(3):
        tr._tc.ppo_backward(*args, **kw)
    times = []
    for _ in range(repeats):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        tr._tc.ppo_backward(*args, **kw)
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e) / 1e3)
    times.sort()
    return times[len(times) // 2], rows.numel()


def learn(n, budget):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    out = []
    for name in ("a2c_reference_hyperparameters", "ppo_defaults"):
        env = VecEnv(n, seed=5, features=True, emit_grids=False)
        torch.manual_seed(0)
        pol = Policy(env.flat_dim, env.n_actions)
        tr = A2CTrainer(env, pol, tensor_cores=True) if name.startswith("a2c") else PPOTrainer(env, pol)
        env.stats(clear=True)
        steps, t0 = 0, time.time()
        reward = torch.zeros((), dtype=torch.float64, device=env.device)
        while steps < budget:
            reward += tr.train_iteration()["mean_reward"].double() * (n * tr.horizon)
            steps += n * tr.horizon
        st = env.stats()
        episodes = max(st["episodes"], 1)
        out.append({"trainer": name, "envs": n, "env_steps": steps, "wall_s": round(time.time() - t0, 1),
                    "mean_episode_reward": float(reward) / episodes, "mean_episode_length": st["steps"] / episodes,
                    "stats": st})
        print(json.dumps(out[-1]), file=sys.stderr, flush=True)
        del tr
        env.close()
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="32768,262144")
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--learn", type=int, default=0, help="env-step budget per trainer for the learning comparison (0: off)")
    ap.add_argument("--learn-envs", type=int, default=32768)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ppo.py measures on a CUDA device; there is none here")
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    res = {"bench": "ppo", "horizon": a.horizon, "epochs": 4, "minibatches": 4, "stepping": "features-only",
           "options": "default", **gpu_info(), "results": []}
    for n in [int(s) for s in a.sizes.split(",")]:
        env = VecEnv(n, seed=1, features=True, emit_grids=False)
        torch.manual_seed(0)
        tr = PPOTrainer(env, Policy(env.flat_dim, env.n_actions), horizon=a.horizon)
        t0 = time.time()
        med, peak, base = time_iterations(tr, a.warmup, a.repeats)
        kt, rows = time_kernel(tr, a.repeats)
        fl = row_flops(env.flat_dim, env.n_actions)
        entry = {"envs": n, "iteration_s": med, "train_env_steps_per_s": n * a.horizon / med,
                 "max_memory_allocated_gb": round(peak / 1e9, 3), "resident_before_iteration_gb": round(base / 1e9, 3),
                 "ppo_kernel_s_per_minibatch": kt, "minibatch_rows": rows, "ppo_kernel_ns_per_row": kt / rows * 1e9,
                 "ppo_kernel_s_per_iteration_computed": kt * tr.epochs * tr.minibatches,
                 "flops_per_row_fp32_network": fl,
                 "ppo_kernel_tflops_fp32_network_six_products_not_counted": fl * rows / kt / 1e12,
                 "wall_s": round(time.time() - t0, 1)}
        res["results"].append(entry)
        print(json.dumps(entry), file=sys.stderr, flush=True)
        del tr
        env.close()
        torch.cuda.empty_cache()
    if a.learn:
        res["learn"] = learn(a.learn_envs, a.learn)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
