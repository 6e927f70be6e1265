"""bench.py prints ONE JSON line with the keys the driver reads (both arms)."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(*args):
    p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, cwd=REPO, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                     # stdout carries the JSON line and nothing else
    return json.loads(lines[0])


def test_reference_arm_line_on_cpu():
    d = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--num-envs", "256")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1
    assert d["metric"] == "env-steps/sec incl. obs" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "lockstep steps" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["timed_lockstep_steps"] >= 512          # never a run so short that it times env creation


@pytest.mark.gpu
def test_gpu_arm_line():
    d = _run("--steps", "64", "--warmup", "3", "--cpu-seconds", "1")
    assert BASE_KEYS | {"clocks", "roofline"} <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 64 and d["warmup"] == 3 and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["value"] > 1e8 and d["gpu_launches"] >= 1 and "workload" in d["config"] and "model" not in d["config"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 4096 and e["d2h_bytes_per_step"] == 4096 * 372
    assert e["value"] < d["value"]                    # host buffers and PCIe inside the timed region
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and cb["single_thread"]["cores"] == 1


@pytest.mark.gpu
def test_gpu_arm_times_exactly_the_given_steps_and_dumps_reproducible_outputs(tmp_path):
    import numpy as np
    import torch
    from wab_gym_b200 import VecEnv
    n, K, W = 4096, 40, 3
    args = ("--steps", str(K), "--warmup", str(W), "--legs", "none", "--skip-e2e", "--skip-cpu")
    runs = [_run(*args, "--dump-outputs", str(tmp_path / d)) for d in ("a", "b")]
    for d in runs:      # the envs stepped W warm-up steps, then the K-step pass twice untimed and once timed
        assert d["steps"] == K and d["episode_stats"]["steps"] == n * (W + 3 * K)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    total = 0
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), name
        total += os.path.getsize(tmp_path / "a" / name)
    assert total <= 64 << 20
    # the dumped step recomputed independently: the same seeded envs and actions through single-step launches
    env = VecEnv(n, seed=0, device="cuda:0")
    gen = torch.Generator(device="cuda:0").manual_seed(1)
    actions = torch.randint(0, env.n_actions, (K + W, n), dtype=torch.uint8, device="cuda:0", generator=gen)
    env.reset()
    for a in list(actions[K:]) + 3 * list(actions[:K]):
        obs, reward, done, info = env.step(a)
    want = {"grids": obs.grids, "food": obs.food, "role": obs.role, "status": obs.status, "reward": reward, "done": done,
            "info": info["info"]}
    want = {k: v.cpu().numpy().astype(np.float32) for k, v in want.items()}
    env.close()
    assert names == sorted([k + ".npy" for k in want] + ["env_index.npy"])
    assert np.array_equal(np.load(tmp_path / "a" / "env_index.npy"), np.arange(n, dtype=np.float64))
    for k, v in want.items():
        assert np.array_equal(np.load(tmp_path / "a" / (k + ".npy")), v), k
