"""Cycles per warp-step of the pipeline kernel's rule warp, by region, at configs[1] (4,096 envs, launches of 256 steps).

Builds the probe library (-DWAB_PIPE_CLOCKS, wab_core.cuh) into a temporary directory, times the default library and the
probe library on the same workload, and prints the launch time of both (so the probe's own cost shows) next to the
probe's table: cycles per warp-step spent in each region of a step, and how many passes per warp-step each rare path
takes. Each library runs in a child process of its own (a process loads one library). Developer tool:
`python tools/pipe_clocks.py [--launches 64] [--out FILE]`."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REGIONS = ["draws", "slide", "deplog", "despawn", "chase", "eat", "tail", "reset", "handoff"]   # PipeRegion order
PATHS = ["steps", "tie", "deplog", "wolves", "eat", "eat_hit", "spawn", "reset"]                 # PipePath order
N, T = 4096, 256


def child(probe, launches, warmup):
    sys.path.insert(0, ROOT)
    os.environ["WAB_PIPE"] = "2"
    import torch
    from wab_gym_b200 import VecEnv
    env = VecEnv(N, seed=1)
    assert "pipe" in env.step_kernel_name(T)
    gen = torch.Generator(device="cuda").manual_seed(1)
    acts = [torch.randint(0, env.n_actions, (T, N), dtype=torch.uint8, device="cuda", generator=gen) for _ in range(4)]
    buf = env._alloc(T)
    env.reset()
    for i in range(warmup):
        env.step_many(acts[i % 4], out=buf)
    read = None
    if probe:
        read = env.lib.wab_pipe_clocks_read
        read.argtypes = [ctypes.c_void_p, ctypes.c_int]
        tot = (ctypes.c_ulonglong * (len(REGIONS) + len(PATHS)))()
        assert read(tot, 1) == 0
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(launches):
        env.step_many(acts[i % 4], out=buf)
    e1.record()
    torch.cuda.synchronize()
    res = {"launch_us": e0.elapsed_time(e1) * 1e3 / launches, "device": torch.cuda.get_device_name()}
    if probe:
        assert read(tot, 0) == 0
        res["cycles"] = dict(zip(REGIONS, list(tot)[:len(REGIONS)]))
        res["paths"] = dict(zip(PATHS, list(tot)[len(REGIONS):]))
    print(json.dumps(res))


def run_child(lib, launches, warmup):
    env = dict(os.environ)
    env.pop("WAB_LIB", None)
    if lib:
        env["WAB_LIB"] = lib
    cmd = [sys.executable, os.path.abspath(__file__), "--child", "--launches", str(launches), "--warmup", str(warmup)]
    if lib:
        cmd.append("--probe")
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, check=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--probe", action="store_true")
    ap.add_argument("--launches", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--out", default=None, help="also write the JSON results here")
    a = ap.parse_args()
    if a.child:
        return child(a.probe, a.launches, a.warmup)
    sys.path.insert(0, ROOT)
    from wab_gym_b200 import build as B
    B.build()
    tmp = tempfile.mkdtemp(prefix="wab_pipe_clocks_")
    lib = os.path.join(tmp, "libwab_b200_clocks.so")
    subprocess.run([B.find_nvcc()] + B.NVCC_FLAGS + ["-DWAB_PIPE_CLOCKS", "-o", lib] + B.SOURCES, check=True,
                   stdout=subprocess.DEVNULL)
    plain = run_child(None, a.launches, a.warmup)
    probe = run_child(lib, a.launches, a.warmup)
    ws = probe["paths"]["steps"]
    print("%s, configs[1]: %d envs, launches of %d steps, pipeline kernel" % (plain["device"], N, T))
    print("launch time: default library %.1f us, probe library %.1f us (%.1f ns vs %.1f ns per step)" % (
        plain["launch_us"], probe["launch_us"], plain["launch_us"] * 1e3 / T, probe["launch_us"] * 1e3 / T))
    total = sum(probe["cycles"].values()) / ws
    print("%-10s %10s %7s" % ("region", "cyc/wstep", "share"))
    for r in REGIONS:
        c = probe["cycles"][r] / ws
        print("%-10s %10.1f %6.1f%%" % (r, c, 100.0 * c / total))
    print("%-10s %10.1f" % ("total", total))
    print("rare paths, passes per warp-step:", " ".join("%s %.4f" % (k, probe["paths"][k] / ws) for k in PATHS[1:]))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump({"default": plain, "probe": probe}, fh, indent=1)


if __name__ == "__main__":
    main()
