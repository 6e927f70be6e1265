#!/usr/bin/env python
"""Build tuning variants of the CUDA library (different -D knobs) and bench each on the GPU box.

    python tools/tune.py [--sizes 4096,1048576] [--steps 256]

Writes one JSON line per (variant, size) to gpurun_out/tune.jsonl. Developer tool; not part of the
product path.
"""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from wab_gym_b200 import build as wab_build  # noqa: E402

VARIANTS = {
    "base": [],
    "mb5": ["-DWAB_MIN_BLOCKS_LPE1=5"],
    "mb8": ["-DWAB_MIN_BLOCKS_LPE1=8"],
    "mb7": ["-DWAB_MIN_BLOCKS_LPE1=7"],
    "cta64": ["-DWAB_THREADS_LPE1=64"],
    "cta32": ["-DWAB_THREADS_LPE1=32"],
    "cta256": ["-DWAB_THREADS_LPE1=256"],
    "slide1": ["-DWAB_SLIDE_UNROLL=1"],
    "slide3": ["-DWAB_SLIDE_UNROLL=3"],
    "spawn1": ["-DWAB_SPAWN_UNROLL=1"],
    "spawn4": ["-DWAB_SPAWN_UNROLL=4"],
    "spawn2": ["-DWAB_SPAWN_UNROLL=2"],
    "spawn3": ["-DWAB_SPAWN_UNROLL=3"],
    "slide2": ["-DWAB_SLIDE_UNROLL=2"],
    "slide6": ["-DWAB_SLIDE_UNROLL=6"],
    "slide2mb5": ["-DWAB_SLIDE_UNROLL=2", "-DWAB_MIN_BLOCKS_LPE1=5"],
    "slide3mb5": ["-DWAB_SLIDE_UNROLL=3", "-DWAB_MIN_BLOCKS_LPE1=5"],
    "s2s2": ["-DWAB_SLIDE_UNROLL=2", "-DWAB_SPAWN_UNROLL=2"],
    "s3s3": ["-DWAB_SLIDE_UNROLL=3", "-DWAB_SPAWN_UNROLL=3"],
    "s2s2mb5": ["-DWAB_SLIDE_UNROLL=2", "-DWAB_SPAWN_UNROLL=2", "-DWAB_MIN_BLOCKS_LPE1=5"],
    "s3s3mb5": ["-DWAB_SLIDE_UNROLL=3", "-DWAB_SPAWN_UNROLL=3", "-DWAB_MIN_BLOCKS_LPE1=5"],
    "s6s6mb4": ["-DWAB_SLIDE_UNROLL=6", "-DWAB_SPAWN_UNROLL=6", "-DWAB_MIN_BLOCKS_LPE1=4"],
    "t32": ["-DWAB_THREADS_LPEN=32"],
    "t128": ["-DWAB_THREADS_LPEN=128"],
    "lpen5": ["-DWAB_MIN_BLOCKS_LPEN=5"],
    "lpen6": ["-DWAB_MIN_BLOCKS_LPEN=6"],
    "lpen8": ["-DWAB_MIN_BLOCKS_LPEN=8"],
    "lpen12": ["-DWAB_MIN_BLOCKS_LPEN=12"],
    "lpen14": ["-DWAB_MIN_BLOCKS_LPEN=14"],
    "s1s1": ["-DWAB_SLIDE_UNROLL=1", "-DWAB_SPAWN_UNROLL=1"],
    "s1s1mb8": ["-DWAB_SLIDE_UNROLL=1", "-DWAB_SPAWN_UNROLL=1", "-DWAB_MIN_BLOCKS_LPE1=8"],
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4096,1048576")
    ap.add_argument("--steps", type=int, default=0,
                    help="timed steps per size; 0: 2^28 env-steps, 256 to 65,536 steps (as tools/window_steps.sh)")
    ap.add_argument("--variants", default=",".join(VARIANTS))
    ap.add_argument("--lpe", default="")
    args = ap.parse_args()
    outdir = os.path.join(REPO, "gpurun_out", "variants")
    os.makedirs(outdir, exist_ok=True)
    results = open(os.path.join(REPO, "gpurun_out", "tune.jsonl"), "a")
    for name in args.variants.split(","):
        lib = os.path.join(outdir, "libwab_%s.so" % name)
        cmd = [wab_build.find_nvcc()] + wab_build.NVCC_FLAGS + VARIANTS[name] + ["-Xptxas", "-v", "-o", lib] + wab_build.SOURCES
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if proc.returncode:
            print(name, "build failed", proc.stdout[-2000:])
            continue
        regs = [l.split("Used ")[1].split(" registers")[0] for l in proc.stdout.splitlines() if "Used" in l]
        for size in args.sizes.split(","):
            for lpe in (args.lpe.split(",") if args.lpe else [""]):
                env = dict(os.environ, WAB_LIB=lib)
                if lpe:
                    env["WAB_LPE"] = lpe
                fuse = 64 if int(size) <= 65536 else 32
                p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--num-envs", size, "--steps", str(args.steps or min(65536, max(256, (1 << 28) // int(size)))),
                                    "--warmup", "8", "--fuse", str(fuse), "--skip-e2e", "--skip-cpu"],
                                   stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
                try:
                    d = json.loads(p.stdout.strip().splitlines()[-1])
                    row = {"variant": name, "lpe": lpe, "n": int(size), "value": d["value"], "per_call": d["per_call"]["value"],
                           "frac": d["roofline"]["frac"], "regs": regs}
                except Exception:
                    row = {"variant": name, "lpe": lpe, "n": int(size), "error": p.stderr[-500:]}
                print(json.dumps(row), flush=True)
                results.write(json.dumps(row) + "\n")
                results.flush()


if __name__ == "__main__":
    main()
