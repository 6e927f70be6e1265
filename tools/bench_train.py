"""Training throughput of A2CTrainer: the tensor-core path (wab_policy_forward collection, torch loss, wab_policy_backward,
Adam) against the torch path (materialised input, cuBLAS forward with autograd, loss.backward()), features-only stepping,
default options. Prints one JSON line (and writes it to --out).

Per size and path: training env-steps/s (one whole iteration = collection + loss + backward + Adam, CUDA events, after
--warmup iterations, median of --repeats), torch.cuda.max_memory_allocated over one iteration. For the tensor-core path
also the backward kernel alone on the last recorded batch (CUDA events, median of --repeats): time per active row and
achieved FLOP/s counted from the shapes — 2 x multiply-adds of the fp32 network (forward recompute, activation and weight
gradients), NOT counting the six bf16 products per fp32 product the tensor cores execute. The torch path is run only where
its autograd footprint (computed from the shapes) fits --torch-max-gb; above that the computed footprint is reported."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:          # the rate is still a measurement; say what could not be read
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unread (%s)" % exc}


def row_flops(dim, n_actions):
    """2 x multiply-adds per active row: forward recompute + activation gradients + weight gradients."""
    fwd = dim * 128 + 128 * 150 + 150 * 128 + 128 * (n_actions + 1)
    act = 128 * 150 + 150 * 128 + 128 * (n_actions + 1)
    return 2 * (fwd + act + fwd)


def torch_footprint_bytes(n, T, dim):
    """What autograd keeps per env-step on the torch path: the input, pre- and post-activations of the three layers,
    the clamp's input and output, the heads' outputs (fp32)."""
    return 4 * n * T * (dim + 2 * (128 + 150 + 128) + 2 * 128 + 16)


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


def time_backward(tr, repeats):
    b, tc = tr.last_batch, tr._tc
    active = ((b["g_logp"] != 0) | (b["g_value"] != 0))
    n_active = int(active.sum())
    rows = torch.nonzero(active.reshape(-1)).squeeze(1).to(torch.int32)
    n_rows = torch.tensor([n_active], dtype=torch.int64, device=rows.device)
    out = torch.empty(tc.n_params, device=rows.device)
    args = (b["features"], b["counters"], b["actions"], b["g_logp"], b["g_value"])
    for _ in range(3):
        tc.backward(*args, out=out, rows=rows, n_rows=n_rows)
    times = []
    for _ in range(repeats):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        tc.backward(*args, out=out, rows=rows, n_rows=n_rows)
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e) / 1e3)
    times.sort()
    return times[len(times) // 2], n_active


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="32768,262144")
    ap.add_argument("--steps", type=int, default=80)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--torch-max-gb", type=float, default=60.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train.py measures on a CUDA device; there is none here")
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.policy import Policy
    res = {"bench": "train", "steps_per_iteration": a.steps, "mode": "episodic", "stepping": "features-only",
           "options": "default", **gpu_info(), "results": []}
    for n in [int(s) for s in a.sizes.split(",")]:
        for tc in (True, False):
            env = VecEnv(n, seed=1, features=True, emit_grids=False)
            entry = {"envs": n, "path": "tensor_cores" if tc else "torch"}
            need = torch_footprint_bytes(n, a.steps, env.flat_dim)
            if not tc:
                entry["autograd_footprint_gb_computed"] = round(need / 1e9, 2)
                if need > a.torch_max_gb * 1e9:
                    entry["skipped"] = "computed footprint above --torch-max-gb"
                    res["results"].append(entry)
                    env.close()
                    continue
            torch.manual_seed(0)
            tr = A2CTrainer(env, Policy(env.flat_dim, env.n_actions), horizon=a.steps, tensor_cores=tc)
            t0 = time.time()
            med, peak, base = time_iterations(tr, a.warmup, a.repeats)
            entry.update({"iteration_s": med, "train_env_steps_per_s": n * a.steps / med,
                          "max_memory_allocated_gb": round(peak / 1e9, 3), "resident_before_iteration_gb": round(base / 1e9, 3),
                          "wall_s": round(time.time() - t0, 1)})
            if tc:
                bt, n_active = time_backward(tr, a.repeats)
                fl = row_flops(env.flat_dim, env.n_actions)
                entry.update({"backward_s": bt, "active_rows": n_active, "backward_ns_per_active_row": bt / max(n_active, 1) * 1e9,
                              "backward_flops_per_row_fp32_network": fl,
                              "backward_tflops_fp32_network_six_products_not_counted": fl * n_active / bt / 1e12})
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
