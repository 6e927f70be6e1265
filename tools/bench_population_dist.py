"""Data-parallel population throughput: one process per GPU (NCCL), world sizes from --worlds (capped at the visible GPU
count), each spawned and joined in turn. PPOPopulation with horizon 64 and 4 epochs x 4 minibatches, default options,
--configs "P x c" per GPU: every rank holds all P members, c envs of each (members of n = world c envs; one blocked
VecEnv of P c envs per rank). Prints one JSON line (and writes it to --out).

Per (world size, config): aggregate collected env-steps/s (world x P x c x horizon over the slowest rank's median
iteration time), each rank's median iteration time (CUDA events, after --warmup iterations, median of --repeats), the
time of one minibatch's cross-rank gradient sum (wab_policy_backward_population_grad_f64 + all-gather of [P, stride] f64 +
wab_policy_grad_sum_ranks) and of its all-gather alone (CUDA events, median of --repeats; at world size 1 the all-gather
is a copy), the bytes each rank sends in it, and the scaling against world size 1. World sizes above the visible GPU
count are reported as not measured."""
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


def _events_time(fn, repeats, skip=3):
    out = []
    for i in range(repeats + skip):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        if i >= skip:
            out.append(s.elapsed_time(e) / 1e3)
    return _median(out)


def _worker(rank, world, port, configs, horizon, warmup, repeats, outdir):
    import torch.distributed as dist
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.population import PPOPopulation
    from wab_gym_b200.sharding import population_shards
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    group = dist.group.WORLD if world > 1 else None
    rows = []
    for P, c in configs:
        n = world * c
        first, cr = population_shards(n, world)[rank]
        env = VecEnv(P * cr, seed=1, features=True, emit_grids=False, env_id_base=first, device=torch.device("cuda", rank),
                     **({"blocks": P, "block_stride": n} if P > 1 else {}))
        torch.manual_seed(0)
        pop = PPOPopulation(env, P, horizon=horizon, group=group)
        for _ in range(warmup):
            pop.train_iteration()
        torch.cuda.synchronize()
        its = []
        for _ in range(repeats):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            pop.train_iteration()
            e.record()
            e.synchronize()
            its.append(s.elapsed_time(e) / 1e3)
        g64 = torch.empty(P, pop._tc.grad_stride, dtype=torch.float64, device=env.device)
        gathered = torch.empty(world, P, pop._tc.grad_stride, dtype=torch.float64, device=env.device)

        def gather():
            dist.all_gather(list(gathered.unbind(0)), g64)

        def grad_sum():
            pop._tc.grad_f64(g64)
            gather()
            pop._tc.grad_sum_ranks(gathered, pop._grad)
        rows.append({"members": P, "envs_per_member_per_gpu": cr, "iteration_s": _median(its),
                     "grad_sum_s_per_minibatch": _events_time(grad_sum, repeats),
                     "all_gather_s_per_minibatch": _events_time(gather, repeats),
                     "all_gather_bytes_sent_per_rank": g64.numel() * 8})
        del pop
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
    ap.add_argument("--worlds", default="1,2,8")
    ap.add_argument("--configs", default="16x2048,4x8192,64x512", help="members x envs per member, per GPU")
    ap.add_argument("--horizon", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_population_dist.py measures on CUDA devices; there is none here")
    configs = [tuple(int(x) for x in cfg.split("x")) for cfg in a.configs.split(",")]
    visible = torch.cuda.device_count()
    res = {"bench": "population_dist", "trainer": "PPOPopulation", "horizon": a.horizon, "epochs": 4, "minibatches": 4,
           "stepping": "features-only", "options": "default", "backend": "nccl", "visible_gpus": visible,
           **gpu_info(), "results": [], "not_measured": []}
    base = {}
    with tempfile.TemporaryDirectory() as tmp:
        for world in (int(w) for w in a.worlds.split(",")):
            if world > visible:
                res["not_measured"].append({"world_size": world, "reason": "only %d GPU(s) visible" % visible})
                continue
            with socket.socket() as s:
                s.bind(("127.0.0.1", 0))
                port = s.getsockname()[1]
            mp.spawn(_worker, args=(world, port, configs, a.horizon, a.warmup, a.repeats, tmp), nprocs=world, join=True)
            with open(os.path.join(tmp, "world%d.json" % world)) as f:
                per_rank = json.load(f)
            for k, (P, c) in enumerate(configs):
                its = [r[k]["iteration_s"] for r in per_rank]
                rate = world * P * c * a.horizon / max(its)
                if world == 1:
                    base[(P, c)] = rate
                entry = {"world_size": world, "members": P, "envs_per_member_per_gpu": c, "collected_env_steps_per_s": rate,
                         "per_rank_iteration_s": its,
                         "per_rank_grad_sum_s_per_minibatch": [r[k]["grad_sum_s_per_minibatch"] for r in per_rank],
                         "per_rank_all_gather_s_per_minibatch": [r[k]["all_gather_s_per_minibatch"] for r in per_rank],
                         "all_gather_bytes_sent_per_rank": per_rank[0][k]["all_gather_bytes_sent_per_rank"],
                         "scaling_vs_world_1": rate / (world * base[(P, c)]) if (P, c) in base else None}
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
