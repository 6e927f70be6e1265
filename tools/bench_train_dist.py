"""Data-parallel PPO throughput: one process per GPU (NCCL), world sizes 1, 2, ... up to --gpus (capped at the visible
GPU count), each spawned and joined in turn. PPOTrainer with horizon 64 and 4 epochs x 4 minibatches, features-only
stepping, default options, --sizes envs PER GPU. Prints one JSON line (and writes it to --out).

Per (world size, size): aggregate collected env-steps/s (world x envs x horizon over the slowest rank's median iteration
time), each rank's median iteration time (CUDA events, after --warmup iterations, median of --repeats), the time of one
minibatch's cross-rank gradient sum (wab_policy_backward_grad_f64 + all-gather + wab_policy_grad_sum_ranks; CUDA events,
median of --repeats; at world size 1 the all-gather is a copy), and the scaling against world size 1. World sizes above
the visible GPU count are reported as not measured."""
import argparse
import json
import os
import socket
import sys
import tempfile

import torch
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.bench_train import gpu_info  # noqa: E402


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def _worker(rank, world, port, sizes, horizon, warmup, repeats, outdir):
    import torch.distributed as dist
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    rows = []
    for n in sizes:
        env = VecEnv(n, seed=1, features=True, emit_grids=False, env_id_base=rank * n, device=torch.device("cuda", rank))
        torch.manual_seed(0)
        tr = PPOTrainer(env, Policy(env.flat_dim, env.n_actions), horizon=horizon, group=dist.group.WORLD if world > 1 else None)
        for _ in range(warmup):
            tr.train_iteration()
        torch.cuda.synchronize()
        its = []
        for _ in range(repeats):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            tr.train_iteration()
            e.record()
            e.synchronize()
            its.append(s.elapsed_time(e) / 1e3)
        g64 = torch.empty(tr._tc.n_params, dtype=torch.float64, device=env.device)
        gathered = torch.empty(world, tr._tc.n_params, dtype=torch.float64, device=env.device)
        red = []
        for i in range(repeats + 3):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            tr._tc.grad_f64(g64)
            dist.all_gather(list(gathered.unbind(0)), g64)
            tr._tc.grad_sum_ranks(gathered, tr._grad)
            e.record()
            e.synchronize()
            if i >= 3:
                red.append(s.elapsed_time(e) / 1e3)
        rows.append({"envs_per_gpu": n, "iteration_s": _median(its), "grad_sum_s_per_minibatch": _median(red)})
        del tr
        env.close()
        torch.cuda.empty_cache()
    out = [None] * world
    dist.all_gather_object(out, rows)
    if rank == 0:
        with open(os.path.join(outdir, "world%d.json" % world), "w") as f:
            json.dump(out, f)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=8)
    ap.add_argument("--sizes", default="32768,262144")
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_dist.py measures on CUDA devices; there is none here")
    sizes = [int(s) for s in a.sizes.split(",")]
    visible = torch.cuda.device_count()
    res = {"bench": "train_dist", "trainer": "PPOTrainer", "horizon": a.horizon, "epochs": 4, "minibatches": 4,
           "stepping": "features-only", "options": "default", "backend": "nccl", "visible_gpus": visible,
           **gpu_info(), "results": [], "not_measured": []}
    base = {}
    with tempfile.TemporaryDirectory() as tmp:
        for world in range(1, a.gpus + 1):
            if world > visible:
                res["not_measured"].append({"world_size": world, "reason": "only %d GPU(s) visible" % visible})
                continue
            with socket.socket() as s:
                s.bind(("127.0.0.1", 0))
                port = s.getsockname()[1]
            mp.spawn(_worker, args=(world, port, sizes, a.horizon, a.warmup, a.repeats, tmp), nprocs=world, join=True)
            with open(os.path.join(tmp, "world%d.json" % world)) as f:
                per_rank = json.load(f)
            for k, n in enumerate(sizes):
                its = [r[k]["iteration_s"] for r in per_rank]
                rate = world * n * a.horizon / max(its)
                if world == 1:
                    base[n] = rate
                entry = {"world_size": world, "envs_per_gpu": n, "collected_env_steps_per_s": rate,
                         "per_rank_iteration_s": its,
                         "per_rank_grad_sum_s_per_minibatch": [r[k]["grad_sum_s_per_minibatch"] for r in per_rank],
                         "scaling_vs_world_1": rate / (world * base[n]) if n in base else None}
                res["results"].append(entry)
                print(json.dumps(entry), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
