"""Cost of any loss through the tensor-core policy (PolicyTrainTC.logits_and_value) against the fused PPO kernel.
Prints one JSON line (and writes it to --out).

Per size (PPO's minibatch: envs x horizon / minibatches rows of a batch collected by PPOTrainer), in one process, CUDA
events, --warmup launches first, median of --repeats:
- eval: wab_policy_evaluate alone (logits and value of the listed rows), ns per row;
- logits_backward: wab_policy_backward_logits alone, the reduction included, ns per row;
- ppo_fused: wab_policy_ppo_backward alone (as tools/bench_ppo.py times it), the reduction included, ns per row;
- minibatch_function: one PPO minibatch through the autograd Function (evaluate, ppo_loss in torch on the logits and
  value, .backward() into the parameters' .grad), against minibatch_fused: the same minibatch as one
  wab_policy_ppo_backward launch. Their ratio is what a loss written in torch costs over the fused kernel."""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.bench_train import gpu_info  # noqa: E402


def median_time(fn, warmup, repeats):
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


def measure(tr, warmup, repeats):
    from wab_gym_b200 import _lib
    from wab_gym_b200.ppo import ppo_loss
    from wab_gym_b200.vec_env import _ptr
    tc, b, dev = tr._tc, tr.last_batch, tr.env.device
    tc.refresh()                                    # both routes on the weights after the iteration's last step
    feats, ctrs = b["features"], b["counters"]
    T, N = feats.shape[:2]
    m = T * N // tr.minibatches
    rows = torch.randperm(T * N, device=dev)[:m].to(torch.int32)
    A = tc.heads[0].shape[0] - 1
    logits, value = torch.empty(m, A, device=dev), torch.empty(m, device=dev)
    g_logits, g_value = torch.randn(m, A, device=dev) * 1e-6, torch.randn(m, device=dev) * 1e-6
    grad = torch.empty(tc.n_params, device=dev)
    w, bh = tc.heads

    def evaluate():
        _lib.check(tc.lib.wab_policy_evaluate(
            tc.env._h, _ptr(feats), T, N, _ptr(ctrs), _ptr(rows), m, _ptr(tc.packed), _ptr(tc.bias), _ptr(tc.packed2),
            _ptr(tc.bias2), 150, _ptr(tc.packed3), _ptr(tc.bias3), _ptr(w), _ptr(bh), A, 0.01, 0.01, -4.0, 4.0,
            _ptr(tc.scratch), tc.scratch.numel(), _ptr(logits), _ptr(value), tc._stream()))

    def logits_backward():
        _lib.check(tc.lib.wab_policy_backward_logits(
            tc.env._h, _ptr(feats), T, N, _ptr(ctrs), _ptr(rows), m, _ptr(g_logits), _ptr(g_value), _ptr(tc.packed),
            _ptr(tc.bias), _ptr(tc.packed2), _ptr(tc.bias2), 150, _ptr(tc.packed3), _ptr(tc.bias3), _ptr(tc.packed2t),
            _ptr(tc.packed3t), _ptr(w), _ptr(bh), A, 0.01, 0.01, -4.0, 4.0, _ptr(tc.scratch), tc.scratch.numel(),
            _ptr(grad), tc._stream()))

    r64 = rows.long()
    a, lp_old = b["actions"].reshape(-1)[r64].long(), b["logp"].reshape(-1)[r64]
    adv, target = b["advantage"].reshape(-1)[r64], b["target"].reshape(-1)[r64]
    count = torch.tensor([m], dtype=torch.int64, device=dev)

    def fused():
        tc.ppo_backward(feats, ctrs, b["actions"], b["logp"], b["advantage"], b["target"], rows, count, tr.clip_eps,
                        1.0 / m, tr.vf_coef / m, tr.ent_coef / m, out=grad)

    def function():
        for p in tr.policy.parameters():
            p.grad = None
        lg, val = tc.logits_and_value(feats, ctrs, rows)
        logq = torch.log_softmax(lg, -1)
        loss, _ = ppo_loss(logq.gather(1, a[:, None]).squeeze(1), val, -(logq.exp() * logq).sum(-1), lp_old, adv, target,
                           tr.clip_eps, tr.vf_coef, tr.ent_coef)
        loss.backward()

    t_eval = median_time(evaluate, warmup, repeats)
    t_lbw = median_time(logits_backward, warmup, repeats)
    t_fused = median_time(fused, warmup, repeats)
    t_fn = median_time(function, warmup, repeats)
    # the two routes give the same gradient up to rounding (reported, not asserted)
    function()
    g_fn = torch.cat([p.grad.reshape(-1) for p in tr.policy.parameters()])
    fused()
    rel = float((g_fn - grad).abs().max() / grad.abs().max())
    return {"rows": m, "eval_ns_per_row": t_eval / m * 1e9, "logits_backward_ns_per_row": t_lbw / m * 1e9,
            "ppo_fused_ns_per_row": t_fused / m * 1e9, "minibatch_function_s": t_fn, "minibatch_fused_s": t_fused,
            "function_over_fused": t_fn / t_fused, "eval_over_fused": t_eval / t_fused,
            "logits_backward_over_fused": t_lbw / t_fused, "grad_max_rel_diff_function_vs_fused": rel}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="32768,262144")
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_policy_autograd.py measures on a CUDA device; there is none here")
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    res = {"bench": "policy_autograd", "horizon": a.horizon, "minibatches": 4, "stepping": "features-only",
           "options": "default", **gpu_info(), "warmup": a.warmup, "repeats": a.repeats, "results": []}
    for n in [int(s) for s in a.sizes.split(",")]:
        env = VecEnv(n, seed=1, features=True, emit_grids=False)
        torch.manual_seed(0)
        tr = PPOTrainer(env, Policy(env.flat_dim, env.n_actions), horizon=a.horizon, minibatches=4)
        t0 = time.time()
        tr.train_iteration()                        # a real batch (features, counters, actions, GAE) under trained weights
        entry = {"envs": n, **measure(tr, a.warmup, a.repeats), "wall_s": round(time.time() - t0, 1)}
        res["results"].append(entry)
        print(json.dumps(entry), file=sys.stderr, flush=True)
        del tr
        env.close()
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
