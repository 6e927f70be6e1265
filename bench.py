#!/usr/bin/env python
"""bench.py — env-steps/s including observation materialisation (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--num-envs E] [--legs all|none|a,b]
                    [--dump-outputs DIR]

A "step" is one lockstep step of the whole batch: every environment advances one turn and its observation
(u8[3,11,11] + food, role, status), reward and done are written to HBM. Workload at N = 1: BASELINE.json
configs[1] — 4,096 lockstep default-grid v1 environments with fused observation output (weak scaling: 4,096 envs
per GPU, global env ids, no data-path collective).

How the headline's timed region is built: reset, W (>= 3) untimed warm-up steps, then a pass of K steps run twice
untimed (eagerly, which loads every kernel it launches, and as the first replay of its CUDA graph), then the graph
replayed once more, timed: the window holds exactly K steps (--steps), so a long window needs a large K; a small one
measures launch latency (at 4,096 envs 20 steps are one 59 us launch). A pass whose outputs fit the 126 MB L2 (at
4,096 envs, up to about 82 steps) rewrites lines the untimed passes have just written, so its stores may stay in the
L2 inside the window; not measured, and at such K the launch latency bounds the run anyway. The actions
are drawn from fixed seeds, so the same arguments give the same inputs and the same outputs on every run
(--dump-outputs DIR writes the outputs of the last timed step). The other legs replay their pass `repeats` times
back to back until the window is at least --leg-window-ms long, their outputs rotating through a ring of buffers
larger than twice the L2 (the headline rotates its launches through up to that many). In every leg the graph keeps
the host from throttling the queue; the window is bracketed by barrier + synchronize on both sides, timed with CUDA
events on the launching stream, max over ranks. The one collective of the data-parallel run — the 64-byte all-reduce
of the episode statistics — is issued during the window on a SIDE stream (wab_gym_b200.sharding.AsyncStatsReducer):
the compute stream never waits for it and nothing is read on the host before the stop event; its latency is
reported as `collective_us`.

Printed JSON (rank 0, one line):
  value        configs[1], device-resident: actions already in HBM, K steps executed by the multi-step kernel in
               launches of <= --fuse steps, every step's outputs written.
  per_call     the same workload as single-step launches (what a policy in the loop gets), CUDA-graph replayed.
  e2e          the C-ABI host-buffer call (wab_vec_step_host_packed): pinned host actions in, every output in
               pinned host memory when the call returns, stream sync per step.
  roofline     dominant kernel of `value` (wab_step_kernel) vs the measured HBM copy bandwidth: `frac` uses the
               ALGORITHMIC 436 B/env-step (SURVEY.md §8d), `frac_dram` the bytes the kernel really moves (ncu).
  legs         the other BASELINE.json configs, each with its own roofline: large_batch (v1, 131,072 envs per GPU =
               the 8-GPU share of 1M), batch_1m (v1, 1,048,576 envs per GPU), v2_config3 (65,536 worlds 20x20),
               v2_config4 (131,072 worlds 64x64 per GPU = the 8-GPU share of configs[3]'s 1,048,576),
               rollout_fp32 (configs[4]: fp32 actor-critic policy in the loop, 32,768 envs per GPU).
  cpu_baseline the oracle's C restatement of the reference step on all host cores (bounded sample), plus the
               same on one thread.
--impl reference times that C restatement alone (the reference itself is pure Python on pandas, ~16 steps/s per
core, and its sources do not travel to the GPU box); rank 0 only, at least 512 lockstep steps.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

B_ALG = 436  # algorithmic bytes per env-step, SURVEY.md §8(d): 363 obs + 8 scalars + 1 action + 2x32 state
METRIC = "env-steps/sec incl. obs"
ALL_LEGS = ("large_batch", "batch_1m", "v2_config3", "v2_config4", "rollout_fp32")
RING_BYTES = 256 << 20   # output ring per leg: > 2 x the 126 MB L2


def workload_name(n):
    tag = "configs[1]: " if n == 4096 else ""
    return "%swab_env v1 default 11x11 viewport, %d lockstep envs per GPU, fused u8 observation output" % (tag, n)


def config_dict(n, world):
    """The workload, in the same words for both arms (the driver compares the two `config`s)."""
    return {"workload": workload_name(n), "num_envs_per_gpu": n, "global_envs": world * n, "parallelism": "dp%d" % world,
            "actions": "uniform 0-4, pre-generated u8[K,N]", "auto_reset": True}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # default: 131,072 timed steps of 4,096 envs, a window of about a quarter of a second on one B200. Other legs read
    # K too: at this default the e2e leg runs its 20,000-step cap, and --impl reference its 2e8 env-step budget
    # (about 48,800 steps at 4,096 envs, some 30 s on 16 host cores).
    ap.add_argument("--steps", type=int, default=131072, help="timed lockstep steps of the headline")
    ap.add_argument("--warmup", type=int, default=64)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--num-envs", type=int, default=4096, help="environments per GPU")
    ap.add_argument("--fuse", type=int, default=256, help="steps per launch of the multi-step kernel")
    ap.add_argument("--leg-window-ms", type=float, default=60.0, help="shortest timed window of every other leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the headline's last timed step to DIR/<name>.npy (rank 0)")
    ap.add_argument("--legs", default="all", help="all | none | comma list of " + ",".join(ALL_LEGS))
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--host-numa", dest="numa", default="auto", choices=["auto", "off"],
                    help="auto: every rank binds its threads and pinned memory to its GPU's NUMA node (sharding.bind_to_gpu_numa)")
    ap.add_argument("--skip-e2e", action="store_true", help="sweeps only: skip the host-buffer leg")
    ap.add_argument("--skip-cpu", action="store_true", help="sweeps only: skip the cpu_baseline leg")
    return ap.parse_args()


def measured_peak():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dram_bytes_per_env_step(n, T):
    """DRAM bytes the step kernel really moves per env-step, from the `ncu --set full` captures under profiles/
    (dram__bytes_read.sum + dram__bytes_write.sum per launch): the multi-step kernel keeps state in registers, so a
    launch writes 372 B per env-step of outputs (363 grid + 9 scalar bytes; every 32-byte sector it touches is
    fully written) and reads 1 action byte; state (38 B + wolves, read and written once per LAUNCH) and the
    read side of partially written sectors add the rest. Table: (n, T) -> bytes per env-step as measured;
    otherwise the model 372 + 1 + 2 * 40 / T, which the captures match within 1 %."""
    table_path = os.path.join(REPO, "profiles", "dram_traffic_table.json")
    try:
        with open(table_path) as fh:
            tab = json.load(fh)
        hit = tab.get("%d,%d" % (n, T))
        if hit:
            return float(hit["bytes_per_env_step"]), "ncu (%s)" % hit["source"]
    except Exception:
        pass
    return 373.0 + 80.0 / T, "model 372 out + 1 action + 2 x 40 state / T (ncu-calibrated, profiles/dram_traffic_table.json)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, window=None):
        """Median SM clock and throttle reasons of the samples taken inside `window` = (t0, t1) wall-clock seconds of
        the timed region (every sample when fewer than two fall inside it)."""
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        rows = [r for (t, r) in self.rows if window is None or window[0] <= t <= window[1] + 0.05]
        if len(rows) < 2:
            rows = [r for (_, r) in self.rows]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, val in zip(names, r[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


_REAL_STDOUT = []     # fd of the process's real stdout once C-level stdout has been pointed at stderr


def emit(text):
    if _REAL_STDOUT:
        sys.stdout.flush()
        os.write(_REAL_STDOUT[0], (text + "\n").encode())
    else:
        print(text, flush=True)


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_run(n_envs, steps, warmup, seed, threads=0, budget_s=None):
    """The oracle's C restatement of the reference step on the host cores (the reference itself is pure
    Python on pandas, ~14-18 steps/s per core in the build container, and cannot travel to this box)."""
    import numpy as np
    from oracle import wab_oracle
    rng = np.random.default_rng(12345)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if threads <= 0:
        threads = cores          # explicit: torchrun exports OMP_NUM_THREADS=1, which must not shrink the CPU arm
    if budget_s is not None:  # bounded sample: size the run from two probes (threads warm on the second)
        rate = 1.0
        for probe_steps in (16, 128):
            a = rng.integers(0, 5, (probe_steps, n_envs)).astype(np.uint8)
            t0 = time.perf_counter()
            wab_oracle.run(None, seed, n_envs, probe_steps, a, threads)
            rate = n_envs * probe_steps / max(time.perf_counter() - t0, 1e-6)
        steps = int(max(8, min(steps, budget_s * rate / n_envs)))
        warmup = 0
    if warmup > 0:
        wab_oracle.run(None, seed, n_envs, warmup, rng.integers(0, 5, (warmup, n_envs)).astype(np.uint8), threads)
    acts = rng.integers(0, 5, (steps, n_envs)).astype(np.uint8)
    t0 = time.perf_counter()
    done_steps, checksum = wab_oracle.run(None, seed, n_envs, steps, acts, threads)
    dt = time.perf_counter() - t0
    return {"value": done_steps / dt, "seconds": dt, "steps": steps, "n_envs": n_envs, "cores": threads,
            "checksum": checksum}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    budget_env_steps = 2.0e8
    n_envs = args.num_envs
    # A timed run of only a few lockstep steps would mostly measure creating and resetting the envs and waking the
    # OpenMP threads, i.e. understate the CPU arm: time at least 512 lockstep steps after at least 16 warm-up steps.
    steps = max(args.steps, 512)
    warmup = max(args.warmup, 16)
    if n_envs * (steps + warmup) > budget_env_steps:
        steps = max(1, int(budget_env_steps / n_envs) - warmup)
    res = cpu_reference_run(n_envs, steps, warmup, args.seed)
    sample = "%d envs x %d lockstep steps (reset on done) after %d warm-up steps, actions uniform 0-4, obs materialised every step" % (
        n_envs, res["steps"], warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "timed_lockstep_steps": res["steps"],
        "ms_per_step": 1e3 * res["seconds"] / res["steps"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 food / integer rules (CPU)",
        "data": "synthetic", "config": config_dict(n_envs, max(world, args.gpus)),
        "cpu_baseline": {"value": res["value"], "unit": "env-steps/s", "cores": res["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": res["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "oracle C port of wab_env.py step+obs with OpenMP over envs, all host threads, one process (whatever --gpus is); "
                "the pandas reference itself: 16.6 steps/s single process, 125 steps/s over 8 cores in the build container "
                "(profiles/r1_reference_cpu_timing.json)",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
class Ctx:
    """Device, process group and the timing discipline shared by every leg."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.numa = None
        if getattr(args, "numa", "auto") == "auto":      # before any pinned allocation: the host-buffer step is host-side bound
            try:
                from wab_gym_b200.sharding import bind_to_gpu_numa
                self.numa = bind_to_gpu_numa(self.local_rank)
            except Exception as exc:
                self.numa = {"error": "%s: %s" % (type(exc).__name__, exc)}
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            # keep stdout to the one JSON line: NCCL prints its version banner on fd 1 (NCCL_DEBUG=VERSION may come from
            # the environment or from a conf file), so C-level stdout goes to stderr and the line is written to the real one
            if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
                os.environ["NCCL_DEBUG"] = "WARN"
            sys.stdout.flush()
            _REAL_STDOUT.append(os.dup(1))
            os.dup2(2, 1)
            dist.init_process_group("nccl", device_id=self.dev)
        self.peak, self.peak_src = measured_peak()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, ms):
        if self.world > 1:
            t = self.torch.tensor([ms], dtype=self.torch.float64, device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def timed_window(self, enqueue, launches_per_unit, min_ms, between=None):
        """Time `repeats` replays of one unit (= `launches_per_unit` calls enqueue(j), captured in a CUDA graph)
        such that the window is >= min_ms, or exactly one replay when min_ms is None. Before the window the unit runs
        once eagerly (loads every kernel, settles every allocation) and, captured, replays untimed (min_ms None: once,
        the first replay uploads the graph; else twice, the calibration). `between(r, repeats)` runs on the host after
        replay r was enqueued (side-stream work only). Returns (window_ms max over ranks, repeats)."""
        torch = self.torch
        side = torch.cuda.Stream(device=self.dev)
        graph = torch.cuda.CUDAGraph()
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for j in range(launches_per_unit):
                enqueue(j)                                    # eager once: warm + every lazy allocation done
            side.synchronize()
            with torch.cuda.graph(graph, stream=side):
                for j in range(launches_per_unit):
                    enqueue(j)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(self.dev)
        e0.record(); graph.replay()
        if min_ms is not None:
            graph.replay()                                              # calibration (also warm-up of the replay)
        e1.record()
        torch.cuda.synchronize(self.dev)
        repeats = 1
        if min_ms is not None:
            unit_ms = self.max_over_ranks(e0.elapsed_time(e1) / 2.0)
            repeats = max(1, int(math.ceil(min_ms / max(unit_ms, 1e-4))))
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        try:                                  # keep the GPU busy ~0.2 ms while the host enqueues the first replays
            torch.cuda._sleep(400_000)
        except Exception:
            pass
        t_wall = time.time()
        start.record()
        for r in range(repeats):
            graph.replay()
            if between is not None:
                between(r, repeats)
        stop.record()
        self.barrier()
        self.last_window = (t_wall, time.time())
        return self.max_over_ranks(start.elapsed_time(stop)), repeats


def v1_fused_leg(ctx, n, K, W, T, min_ms, with_collective, dump_dir=None):
    """K lockstep steps of n v1 envs per pass through wab_vec_step_many (launches of <= T steps), replayed until the
    window is >= min_ms; min_ms None: one pass, exactly K timed steps. dump_dir: see dump_step_outputs."""
    torch = ctx.torch
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.sharding import AsyncStatsReducer
    env = VecEnv(n, seed=ctx.args.seed, device=ctx.dev, env_id_base=ctx.rank * n)
    once = min_ms is None
    # Launches of <= T steps. K >= T: a pass of K steps is cut into chunks of T. K < T, replayed: a launch carries
    # m = T // K whole passes (the K steps replayed m times inside ONE launch of the multi-step kernel, actions differing
    # per pass).
    m = max(1, T // K) if K < T and not once else 1
    L = m * K if K < T else T                                             # steps per full launch
    chunks = [(s, min(L, m * K - s)) for s in range(0, m * K, L)]         # launches of one unit of m passes
    slots = max(1, int(math.ceil(RING_BYTES / float(L * n * 372))))       # output ring > 2 x L2
    units = 1 if once else max(1, int(math.ceil(slots / float(len(chunks)))))   # units per graph
    slots = min(slots, units * len(chunks))                               # one pass: as many buffers as it has launches
    passes = units * m
    ring = [env._alloc(L) for _ in range(slots)]
    gen = torch.Generator(device=ctx.dev).manual_seed(1 + ctx.rank)
    actions = torch.randint(0, env.n_actions, (passes * K + W, n), dtype=torch.uint8, device=ctx.dev, generator=gen)
    env.reset()
    for s in range(0, W, L):                                              # W untimed warm-up steps
        c = min(L, W - s)
        env.step_many(actions[passes * K + s:passes * K + s + c], out={k: v[:c] for k, v in ring[0].items()})
    launches = [(u * m * K + s, c) for u in range(units) for (s, c) in chunks]

    def enqueue(j):
        s, c = launches[j]
        buf = ring[j % slots]
        env.step_many(actions[s:s + c], out={k: v[:c] for k, v in buf.items()})

    reducer = AsyncStatsReducer(ctx.dev) if with_collective else None

    def between(r, repeats):           # SURVEY §8(e): the statistics all-reduce, every few launches, on a side stream
        if r % max(1, repeats // 16) == 0:
            reducer.submit(env.stats_tensor)

    if reducer is not None:
        reducer.submit(env.stats_tensor)                                  # NCCL sets its channels up on first use
        reducer.result()
    window_ms, repeats = ctx.timed_window(enqueue, len(launches), min_ms, between=between if reducer is not None else None)
    if dump_dir is not None and ctx.rank == 0:
        dump_step_outputs(dump_dir, ring[(len(launches) - 1) % slots], launches[-1][1] - 1)
    total_steps = repeats * passes * K
    n_launch = repeats * len(launches)
    collective_us = None
    stats_all = None
    if reducer is not None:
        reducer.submit(env.stats_tensor)
        stats_all = reducer.result()                                      # host read AFTER the stop event
        if ctx.world > 1:
            t = env.stats_tensor()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            samples = []
            for _ in range(5):
                torch.cuda.synchronize(ctx.dev)
                e0.record(); ctx.dist.all_reduce(t); e1.record()
                torch.cuda.synchronize(ctx.dev)
                samples.append(e0.elapsed_time(e1) * 1e3)
            collective_us = sorted(samples)[2]
    stats = env.stats()
    kernel_name = env.step_kernel_name(int(round(total_steps / n_launch)))
    env.close()
    del ring
    torch.cuda.empty_cache()
    per_launch_ms = window_ms / n_launch
    steps_per_launch = total_steps / n_launch
    achieved = B_ALG * n * total_steps / (window_ms * 1e-3) / 1e9
    bpe, bpe_src = dram_bytes_per_env_step(n, int(round(steps_per_launch)))
    roof = {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
            "traffic": bpe * n * steps_per_launch, "traffic_source": bpe_src,
            "frac_dram": achieved / B_ALG * bpe / ctx.peak,
            "kernel": kernel_name, "peak_source": ctx.peak_src,
            "bytes_per_env_step": B_ALG, "dram_bytes_per_env_step": bpe, "env_steps_per_launch": n * steps_per_launch,
            "avg_launch_ms": per_launch_ms,
            "how": "algorithmic bytes of all launches of the timed window / the window (CUDA events on the launching stream; "
                   "launches are back to back in a graph, so inter-launch gaps count against the kernel)"}
    return {"value": ctx.world * n * total_steps / (window_ms * 1e-3), "unit": "env-steps/s", "window_ms": window_ms,
            "repeats": repeats * passes, "steps_per_pass": K, "steps_per_launch": steps_per_launch, "launches": n_launch,
            "ms_per_step": window_ms / total_steps, "num_envs_per_gpu": n, "global_envs": ctx.world * n,
            "ring": "%d output buffers of %d MB (ring of %d MB; the L2 holds 126 MB), rotated per launch" % (
                slots, int(L * n * 372 / 1e6), int(slots * L * n * 372 / 1e6)),
            "roofline": roof, "collective_us": collective_us,
            "collectives_in_window": (reducer.submitted - 2) if reducer is not None else 0,
            "episode_stats": stats_all or stats}


DUMP_MAX_ENVS = 32768       # x 369 float32 values per env = 48 MB, under the 64 MB a dump may take


def dump_step_outputs(path, buf, t):
    """Write step t of the multi-step output buffer `buf` — what a caller of wab_vec_step_many receives for that step:
    grids, food, role, status, reward, done, info — as float32 DIR/<name>.npy, for at most DUMP_MAX_ENVS envs (a fixed,
    seeded sample of them when there are more). env_index.npy (float64) holds the envs' indices."""
    import numpy as np
    import torch
    n = buf["food"].shape[1]
    idx = np.arange(n)
    if n > DUMP_MAX_ENVS:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ENVS, replace=False))
    sel = torch.from_numpy(idx).to(buf["food"].device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))
    for name, v in buf.items():
        if v is not None:
            np.save(os.path.join(path, name + ".npy"), v[t].index_select(0, sel).cpu().numpy().astype(np.float32))


def v1_percall_leg(ctx, n, K, W, min_ms):
    """Single-step launches (what a policy in the loop gets), G of them per CUDA graph."""
    torch = ctx.torch
    from wab_gym_b200 import VecEnv
    env = VecEnv(n, seed=ctx.args.seed, device=ctx.dev, env_id_base=ctx.rank * n)
    G = max(1, min(64, K))
    gen = torch.Generator(device=ctx.dev).manual_seed(101 + ctx.rank)
    actions = torch.randint(0, env.n_actions, (G, n), dtype=torch.uint8, device=ctx.dev, generator=gen)
    env.reset()
    for t in range(W):
        env.step(actions[t % G])
    window_ms, repeats = ctx.timed_window(lambda j: env.step(actions[j]), G, min_ms)
    lpe = env.lanes_per_env
    env.close()
    steps = repeats * G
    achieved = B_ALG * n * steps / (window_ms * 1e-3) / 1e9
    return {"value": ctx.world * n * steps / (window_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": window_ms / steps,
            "window_ms": window_ms, "launches": steps,
            "mode": "1 launch per step, %d-step CUDA graph replayed %d times (actions repeat per replay; outputs "
                    "rewritten in place: %d KB per step, L2-resident)" % (G, repeats, n * 372 // 1024),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
                         "kernel": "wab_step_kernel<false, LPE=%d>, 1 step per launch" % lpe}}


def v2_leg(ctx, n, dims, min_ms, name):
    """Environment 2.0 world turns (SURVEY §8 a16-a18): n lockstep worlds per GPU, contiguous world-id shards."""
    torch = ctx.torch
    from wab_gym_b200.world2 import VecWorld2
    Wd, Hd, no, nw, nb = dims
    A, E = no + nw, no + nw + nb
    env = VecWorld2(n, Wd, Hd, no, nw, nb, seed=ctx.args.seed, env_id_base=ctx.rank * n, device=ctx.dev)
    env.reset_environment()
    gen = torch.Generator(device=ctx.dev).manual_seed(7 + ctx.rank)
    acts = torch.empty((8, A, n), dtype=torch.uint8, device=ctx.dev)       # entity-major, like every v2 array
    acts[:, :no] = torch.randint(0, 6, (8, no, n), dtype=torch.uint8, device=ctx.dev, generator=gen)
    acts[:, no:] = torch.randint(0, 5, (8, nw, n), dtype=torch.uint8, device=ctx.dev, generator=gen)
    for t in range(3):
        env.turn(acts[t])
    window_ms, repeats = ctx.timed_window(lambda j: env.turn(acts[j]), 8, min_ms)
    turns = repeats * 8
    S = 2 * env.R + 1
    bytes_per_turn = A * (3 * S * S + 9) + 2 * E * 8
    kernel = env.kernel_name() if hasattr(env, "kernel_name") else "wab2 turn kernel"
    traffic, traffic_src = None, None
    try:                      # DRAM bytes of one launch (= one turn of all worlds) as ncu measured them, scaled to this batch
        with open(os.path.join(REPO, "profiles", "dram_traffic_table.json")) as fh:
            hit = json.load(fh).get("v2_config3" if name.startswith("configs[2]") else "v2_config4")
        if hit:
            traffic, traffic_src = float(hit["bytes_per_world_turn"]) * n, "ncu (%s)" % hit["source"]
    except Exception:
        pass
    env.close()
    del env
    torch.cuda.empty_cache()
    tps = n * turns / (window_ms * 1e-3)
    achieved = tps * bytes_per_turn / 1e9
    return {"workload": "%s: Environment 2.0 World(%d,%d), %d ostriches %d wolves %d bushes, %d lockstep worlds per GPU" % (
                name, Wd, Hd, no, nw, nb, n),
            "value": ctx.world * tps, "unit": "world-turns/s", "entity_steps_per_s": ctx.world * tps * E,
            "ms_per_turn": window_ms / turns, "window_ms": window_ms, "turns": turns, "launches": turns,
            "num_worlds_per_gpu": n, "global_worlds": ctx.world * n,
            "outputs": "per acting entity a %dx%dx3 u8 window + 5 int32 + reward + done, rewritten per turn (%d MB > L2)" % (
                S, S, int(A * n * 3 * S * S / 1e6)),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
                         "bytes_per_world_turn": bytes_per_turn, "kernel": kernel, "traffic": traffic, "traffic_source": traffic_src,
                         "frac_dram": (tps * traffic / n / 1e9 / ctx.peak) if traffic else None}}


def rollout_leg(ctx, n, K, min_ms):
    """configs[4]: the reference's actor-critic policy (actor_critic.py:54-97), fp32, consuming device-resident
    observations: features -> policy -> Categorical sample -> env.step, nothing leaves the GPU."""
    torch = ctx.torch
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy, Rollout
    torch.manual_seed(0)
    env = VecEnv(n, seed=ctx.args.seed, device=ctx.dev, env_id_base=ctx.rank * n, features=True)
    ro = Rollout(env, Policy(env.flat_dim, env.n_actions), use_graph=True, dtype=torch.float32)
    ro.run(10)
    torch.cuda.synchronize(ctx.dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); ro.run(8); e1.record()
    torch.cuda.synchronize(ctx.dev)
    step_ms = ctx.max_over_ranks(e0.elapsed_time(e1) / 8.0)
    steps = max(K if K <= 512 else 512, int(math.ceil(min_ms / max(step_ms, 1e-4))))
    ctx.barrier()
    e0.record(); ro.run(steps); e1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    st = env.stats()
    desc = ro.describe() if hasattr(ro, "describe") else "flatten+noise kernel -> torch fp32 MLP (cuBLAS) -> sampling kernel -> wab_step_kernel"
    tc = bool(getattr(ro, "tc_trunk", False))
    env.close()
    # the same loop with the policy as library calls (flatten kernel -> three cuBLAS fp32 GEMMs -> tail kernel), for comparison
    lib = None
    if tc:
        env2 = VecEnv(n, seed=ctx.args.seed, device=ctx.dev, env_id_base=ctx.rank * n, features=True)
        ro2 = Rollout(env2, Policy(env2.flat_dim, env2.n_actions), use_graph=True, dtype=torch.float32, tc_first_layer=False, tc_trunk=False)
        ro2.run(10)
        ctx.barrier()
        s2 = max(32, steps // 4)
        e0.record(); ro2.run(s2); e1.record()
        ctx.barrier()
        ms2 = ctx.max_over_ranks(e0.elapsed_time(e1))
        lib = {"value": ctx.world * n * s2 / (ms2 * 1e-3), "ms_per_step": ms2 / s2, "steps": s2, "path": ro2.describe()}
        env2.close()
    # and with FEATURES-ONLY stepping (VecEnv(emit_grids=False)): the policy consumes the 28 feature bytes, so the 363-byte
    # one-hot grids need not be materialised in HBM at all — reported beside the headline, which writes them
    fo = None
    try:
        env3 = VecEnv(n, seed=ctx.args.seed, device=ctx.dev, env_id_base=ctx.rank * n, features=True, emit_grids=False)
        ro3 = Rollout(env3, Policy(env3.flat_dim, env3.n_actions), use_graph=True, dtype=torch.float32)
        ro3.run(10)
        ctx.barrier()
        e0.record(); ro3.run(steps); e1.record()
        ctx.barrier()
        ms3 = ctx.max_over_ranks(e0.elapsed_time(e1))
        fo = {"value": ctx.world * n * steps / (ms3 * 1e-3), "ms_per_step": ms3 / steps, "steps": steps,
              "path": "same loop, wab_step_kernel with d_grids = NULL: features, scalars, reward, done, info only"}
        env3.close()
    except Exception as exc:
        fo = {"error": "%s: %s" % (type(exc).__name__, exc)}
    flops = 2.0 * (env.flat_dim * 128 + 128 * 150 + 150 * 128 + 128 * (env.n_actions + 1))
    v = n * steps / (ms * 1e-3)
    return {"workload": "configs[4]: actor_critic.py rollout, policy %d-128-150-128-{%d,1} fp32 in the loop, %d v1 envs per GPU" % (
                env.flat_dim, env.n_actions, n),
            "value": ctx.world * v, "unit": "env-steps/s", "ms_per_step": ms / steps, "window_ms": ms, "steps": steps,
            "dtype": ("fp32 policy (fp32-accurate on the tensor cores: bf16 x 3 operand splits, fp32 accumulation; "
                      "tests/test_rollout_gpu.py holds it to 3e-6 of the fp64 result)") if tc else "fp32 policy",
            "num_envs_per_gpu": n, "global_envs": ctx.world * n, "path": desc, "library_path": lib, "features_only": fo,
            "policy_flops_per_env_step": flops, "policy_tflops": v * flops / 1e12,
            "mean_episode_length": st["steps"] / max(st["episodes"], 1)}


def e2e_leg(ctx, n, K, W):
    """K (at least 100 ms worth of) steps through the host-buffer C-ABI call, host copies inside the timed region."""
    torch = ctx.torch
    from wab_gym_b200 import VecEnv
    env = VecEnv(n, seed=ctx.args.seed, device=ctx.dev, env_id_base=ctx.rank * n)
    gen = torch.Generator(device=ctx.dev).manual_seed(1 + ctx.rank)
    hb = env.alloc_host_buffers(pinned=True)
    host_actions = torch.randint(0, env.n_actions, (256, n), dtype=torch.uint8, device=ctx.dev, generator=gen).cpu().pin_memory()
    env.reset_host(hb)
    acts_np, hnp = host_actions.numpy(), hb["np"]     # numpy views of the pinned buffers: no per-step torch dispatch
    for t in range(max(W, 8)):
        hnp["actions"][:] = acts_np[t % 256]
        env.step_host(hb)
    t0 = time.perf_counter()
    for t in range(16):
        hnp["actions"][:] = acts_np[t]
        env.step_host(hb)
    per = (time.perf_counter() - t0) / 16
    Ke = int(min(max(K, math.ceil(0.1 / per)), 20000))
    ctx.barrier()
    t0 = time.perf_counter()
    acc = 0.0
    for t in range(Ke):
        hnp["actions"][:] = acts_np[t & 255]     # this step's inputs, host memory
        env.step_host(hb)
        acc += float(hnp["reward"][0])           # the step's result is read on the host
    torch.cuda.synchronize(ctx.dev)
    mine_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = ctx.max_over_ranks(mine_ms)
    per_rank, numa = None, [ctx.numa]
    if ctx.world > 1:
        t = torch.zeros(ctx.world, dtype=torch.float64, device=ctx.dev)
        t[ctx.rank] = n * Ke / (mine_ms * 1e-3)
        ctx.dist.all_reduce(t)
        per_rank = [float(x) for x in t.cpu()]
        numa = [None] * ctx.world
        ctx.dist.all_gather_object(numa, ctx.numa)
    mapped = n <= 16384
    env.close()
    return {"value": ctx.world * n * Ke / (e2e_ms * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": n,
            "d2h_bytes_per_step": n * (363 + 1 + 1 + 1 + 4 + 1 + 1), "steps": Ke, "ms_per_step": e2e_ms / Ke,
            "per_rank": per_rank, "numa": numa,
            "path": ("wab_vec_step_host_packed, <= 16,384 envs: wab_step_kernel reads the pinned host actions and streams grids/food/"
                     "role/status/reward/done/info straight into the pinned host block over PCIe -> stream sync" if mapped else
                     "wab_vec_step_host_packed: pinned host actions -> H2D -> wab_step_kernel -> one D2H of grids/food/role/status/"
                     "reward/done/info into a pinned block -> stream sync")}


def run_ours(args):
    ctx = Ctx(args)
    torch = ctx.torch
    n, K, W, T = args.num_envs, args.steps, max(args.warmup, 3), max(1, args.fuse)
    want = ALL_LEGS if args.legs == "all" else tuple(x for x in args.legs.split(",") if x in ALL_LEGS)

    with ClockSampler(ctx.local_rank) as clocks:
        main = v1_fused_leg(ctx, n, K, W, T, None, with_collective=True, dump_dir=args.dump_outputs)
        main_window = ctx.last_window
    percall = v1_percall_leg(ctx, n, K, W, args.leg_window_ms)

    legs = {}
    # the big-batch legs bound their output buffer: <= 128 steps per launch at 131,072 envs (6.2 GB), <= 24 at 1M envs (9.4 GB)
    plan = {
        "large_batch": lambda: v1_fused_leg(ctx, 131072, min(K, 128), W, 128, args.leg_window_ms, with_collective=False),
        "batch_1m": lambda: v1_fused_leg(ctx, 1048576, min(K, 24), W, 24, args.leg_window_ms, with_collective=False),
        "v2_config3": lambda: v2_leg(ctx, 65536, (20, 20, 10, 3, 20), args.leg_window_ms, "configs[2]"),
        "v2_config4": lambda: v2_leg(ctx, 131072, (64, 64, 8, 64, 256), args.leg_window_ms, "configs[3] (8-GPU share of 1,048,576)"),
        "rollout_fp32": lambda: rollout_leg(ctx, 32768, K, args.leg_window_ms),
    }
    for name in want:
        try:
            legs[name] = plan[name]()
            if name in ("large_batch", "batch_1m"):
                legs[name]["workload"] = workload_name(legs[name]["num_envs_per_gpu"])
        except Exception as exc:      # a leg must never take the headline down with it
            legs[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            try:
                torch.cuda.synchronize(ctx.dev)
                torch.cuda.empty_cache()
            except Exception:
                pass

    e2e = None if args.skip_e2e else e2e_leg(ctx, n, K, W)

    if ctx.rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": "env-steps/s", "n_gpus": ctx.world,
            "steps": K, "warmup": W, "repeats": main["repeats"], "window_ms": main["window_ms"],
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8 grids / int32 rules / u32 Philox (int food counter proven == f64)",
            "data": "synthetic", "config": config_dict(n, ctx.world),
            "timing": {"mode": "wab_vec_step_many, %g steps per launch, every step's obs/reward/done written; the K = %d steps "
                               "timed once, a %.3g ms window" % (main["steps_per_launch"], K, main["window_ms"]),
                       "l2": main["ring"] + "; state lives in registers, no reuse between steps",
                       "collective": "64-byte statistics all-reduce on a side stream, %d issued inside the window, none awaited "
                                     "before the stop event" % main["collectives_in_window"]},
            "clocks": clocks.summary(main_window),
            "e2e": e2e,
            "per_call": percall,
            "gpu_launches": main["launches"],
            "collective_us": main["collective_us"],
            "roofline": main["roofline"],
            "legs": legs,
            "episode_stats": main["episode_stats"],
        }
        try:
            if args.skip_cpu:
                raise RuntimeError("skipped (--skip-cpu)")
            cb = cpu_reference_run(n, 10 ** 9, 4, args.seed, budget_s=args.cpu_seconds)
            line["cpu_baseline"] = {"value": cb["value"], "unit": "env-steps/s", "cores": cb["cores"], "kind": "port",
                                    "sample": "%d envs x %d lockstep steps, %.1f s of %d-thread CPU work" % (
                                        cb["n_envs"], cb["steps"], cb["seconds"], cb["cores"])}
            one = cpu_reference_run(n, 10 ** 9, 4, args.seed, threads=1, budget_s=min(3.0, args.cpu_seconds))
            line["cpu_baseline"]["single_thread"] = {"value": one["value"], "unit": "env-steps/s", "cores": 1,
                                                     "sample": "%d envs x %d lockstep steps, %.1f s" % (one["n_envs"], one["steps"], one["seconds"])}
            line["cpu_baseline"]["pandas_reference"] = ("the pandas reference itself, timed in the build container: 16.6 steps/s "
                                                        "single process, 125 steps/s over 8 cores (profiles/r1_reference_cpu_timing.json)")
        except Exception as exc:  # the oracle is test infrastructure; its absence must not hide the GPU numbers
            line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": 0, "kind": "port", "sample": "failed: %s" % exc}
        emit(json.dumps(line))
    if ctx.world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
