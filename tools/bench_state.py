"""Time checkpointing on the device: wab_vec_save_state, wab_vec_load_state with observation re-emission, and the
device-to-host copy of VecEnv.state_dict(), for default-option batches caught mid-episode (after 40 random steps).

    python tools/bench_state.py [--sizes 131072,1048576] [--repeats 20] [--out PATH]

Kernel times are CUDA events around each call (after warm-up), the state_dict time is a host clock around a call that
ends in a synchronise. Bytes are counted from the record size, the slab columns each kernel touches (only live wolf and
log slots) and the 3 x 11 x 11 + 3 observation bytes per env the load's re-emission writes. Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from wab_gym_b200 import VecEnv, _lib  # noqa: E402
from wab_gym_b200.vec_env import _ptr  # noqa: E402

# per-env bytes of the [N] columns: pos 4, misc 4, nlog 2, episode 4, bkey 8, window 16 (+ food 8 in F64 mode)
FIXED_COLUMNS = 4 + 4 + 2 + 4 + 8 + 16
OBS_BYTES = 3 * 11 * 11 + 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
    except Exception as exc:  # the figure is reported without it rather than guessed
        name, power = torch.cuda.get_device_name(0), "unknown (%s)" % exc
    return {"gpu": name, "power_limit": power}


def time_events(fn, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e-3)
    return times


def bench(n, repeats):
    env = VecEnv(n, seed=1)
    lib, h = env.lib, env._h
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(40):
        env.step(torch.randint(0, env.n_actions, (n,), dtype=torch.uint8, device="cuda", generator=g))
    R = env.record_bytes
    records = torch.empty((n, R), dtype=torch.uint8, device="cuda")
    rejected = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = env._stream()
    obs = env._obs_struct(env._out)
    env._bind(env._out)

    def save():
        _lib.check(lib.wab_vec_save_state(h, None, n, _ptr(records), stream))

    def load():
        _lib.check(lib.wab_vec_load_state(h, _ptr(records), None, n, obs, _ptr(rejected), stream))

    before = env.export_state()
    t_save = time_events(save, repeats)
    t_load = time_events(load, repeats)
    assert int(rejected.item()) == 0
    after = env.export_state()
    assert all(np.array_equal(before[k], after[k]) for k in before), "save/load changed the state"

    host = records.cpu().numpy()
    live_wolves = int(host[:, 52:56].copy().view(np.uint32).sum())
    live_log = int(host[:, 72:76].copy().view(np.uint32).sum())
    f64 = 8 if env.game.food_mode == 0 else 0
    columns = n * (FIXED_COLUMNS + f64) + 4 * live_wolves + 5 * live_log
    save_bytes = columns + n * R
    # load: records in, columns out; then the reset kernel reads and stores the columns it keeps (all but the log)
    # and writes the observation
    reset_columns = n * (FIXED_COLUMNS + f64 + 4) + 4 * live_wolves
    load_bytes = n * R + columns + 2 * reset_columns + n * OBS_BYTES

    torch.cuda.synchronize()
    t_sd = []
    for i in range(repeats + 2):
        t0 = time.perf_counter()
        sd = env.state_dict()
        t1 = time.perf_counter()
        if i >= 2:
            t_sd.append(t1 - t0)
    del sd
    med = lambda v: float(np.median(v))
    out = {
        "envs": n, "record_bytes": R, "repeats": repeats, "live_wolves": live_wolves, "live_log_entries": live_log,
        "save": {"median_s": med(t_save), "min_s": min(t_save), "bytes": save_bytes, "GB_per_s": save_bytes / med(t_save) / 1e9},
        "load_with_obs": {"median_s": med(t_load), "min_s": min(t_load), "bytes": load_bytes,
                          "GB_per_s": load_bytes / med(t_load) / 1e9},
        "state_dict_to_host": {"median_s": med(t_sd), "min_s": min(t_sd), "record_bytes_total": n * R,
                               "GB_per_s": n * R / med(t_sd) / 1e9},
    }
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="131072,1048576")
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_state needs a CUDA device")
    res = {"tool": "tools/bench_state.py", **card(), "cuda_device": torch.cuda.get_device_name(0),
           "results": [bench(int(s), args.repeats) for s in args.sizes.split(",")]}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
