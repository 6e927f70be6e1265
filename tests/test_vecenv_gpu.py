"""Parity tests proper: the CUDA path, called through the C ABI, against the oracle and the
reference traces. Bit-exact for grids, food, role, status, done, positions, wolves; reward compared
as the f32 image of the reference's float64 sum (tolerance 0)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import wab_oracle
from oracle.wab_oracle import OracleEnv
from tests.util import (OPTION_SETS, golden_names, golden_wolves, load_golden, mask_words_to_int, pick_action,
                        window_mask_from_bushes)

pytestmark = pytest.mark.gpu


def _vec(*a, **k):
    from wab_gym_b200 import VecEnv
    return VecEnv(*a, **k)


def _wolves(st, i):
    return sorted((int(a), int(b)) for a, b in st["wolves"][i][: st["n_wolves"][i]])


@pytest.mark.parametrize("name", golden_names())
def test_compat_env_reproduces_reference_trace(name):
    """Single-env gym surface (no auto-reset, fp64 food) vs the REAL reference's recorded trace."""
    from wab_gym_b200 import WolvesAndBushesEnv, default_game_options
    meta, tr = load_golden(name)
    opts = {**default_game_options, **meta["overrides"]}
    env = WolvesAndBushesEnv(opts, seed=meta["seed"], env_id=meta["env_id"])
    assert env.action_space.n == meta["n_actions"]
    vec_state = None
    for t in range(len(tr["action"])):
        a = int(tr["action"][t])
        if t == 0:
            obs, reward, done = env._get_obs(), 0.0, False      # the reset inside the constructor
        elif a < 0:
            obs, reward, done = env.reset(), 0.0, False
        else:
            obs, reward, done, info = env.step(a)
            assert info == {}
        assert len(obs) == 7 and obs[0].dtype == np.float64 and obs[0].shape == (11, 11)
        for p in range(3):
            assert np.array_equal(obs[p], tr["grids"][t][p].astype(np.float64)), (name, t, p)
        assert (obs[3], obs[4], obs[5]) == (tr["food"][t], tr["role"][t], tr["status"][t]), (name, t)
        assert reward == tr["reward"][t] and done == bool(tr["done"][t]), (name, t, reward)
    with pytest.raises(IndexError):
        env.step(env.action_space.n)
    env.close()


@pytest.mark.parametrize("name", sorted(OPTION_SETS))
@pytest.mark.parametrize("f64", [False, True])
def test_vecenv_matches_oracle_per_env(name, f64):
    """N = 70 (two full warps + a ragged one) lockstep envs vs 70 oracle envs, every step, hidden state too."""
    overrides, greedy = OPTION_SETS[name]
    n, steps, seed, base = 70, 260, 5, 1000
    env = _vec(n, overrides, seed=seed, env_id_base=base, force_f64_food=f64, wolf_cap=64)
    oracles = [OracleEnv(overrides, seed=seed, env_id=base + i) for i in range(n)]
    rng = np.random.default_rng(11)
    obs = env.reset()
    cur = [o.reset() for o in oracles]

    def compare(tag, reward=None, done=None, want_r=None, want_d=None):
        g, f, r, s = (t.cpu().numpy() for t in obs)
        st = env.export_state()
        for i, o in enumerate(oracles):
            assert np.array_equal(g[i], cur[i][0]), (tag, i, np.argwhere(g[i] != cur[i][0]))
            assert (int(f[i]), int(r[i]), int(s[i])) == cur[i][1:], (tag, i)
            hs = o.hidden_state()
            assert (st["x"][i], st["y"][i], st["turn"][i], st["episode"][i]) == (hs["x"], hs["y"], hs["turn"], hs["episode"]), (tag, i)
            assert _wolves(st, i) == hs["wolves"], (tag, i)
            assert mask_words_to_int(st["bush_mask"][i]) == window_mask_from_bushes(hs), (tag, i)
            if env.game.food_mode == 0:
                assert st["food"][i] == hs["food"], (tag, i)
        if reward is not None:
            assert np.array_equal(reward, want_r) and np.array_equal(done, want_d), tag

    compare("reset")
    n_done = n_eat = 0
    for t in range(steps):
        acts = np.array([pick_action(rng, cur[i][0], env.n_actions, greedy) for i in range(n)], dtype=np.uint8)
        obs, reward, done, info = env.step(torch.from_numpy(acts).cuda())
        want_r, want_d = np.zeros(n, np.float32), np.zeros(n, bool)
        for i, o in enumerate(oracles):
            c, r, d = o.step(int(acts[i]))
            want_r[i], want_d[i] = np.float32(r), d
            cur[i] = o.reset() if d else c
        compare(("step", t), reward.cpu().numpy(), done.cpu().numpy(), want_r, want_d)
        n_done += int(want_d.sum())
        n_eat += int(((info["info"].cpu().numpy() >> 2) & 1).sum())
    s = env.stats()
    assert s["steps"] == n * steps and s["episodes"] == n_done and s["eats"] == n_eat
    assert s["finished"] + s["starved"] + s["killed"] == n_done and s["bad_actions"] == 0 and s["overflows"] == 0
    env.close()


@pytest.mark.parametrize("lpe", [1, 4, 8, 16, 32])
@pytest.mark.parametrize("name", ["defaults", "dense", "six_actions_random_start"])
def test_every_lanes_per_env_variant_matches_oracle(lpe, name, monkeypatch):
    """The kernel is compiled for 1/4/8/16/32 lanes per env (picked from the batch size); force each
    variant and compare with the oracle. N = 41 leaves a ragged last CTA / warp in every geometry."""
    monkeypatch.setenv("WAB_LPE", str(lpe))
    overrides, greedy = OPTION_SETS[name]
    n, steps, seed, base = 41, 160, 77, 5000
    env = _vec(n, overrides, seed=seed, env_id_base=base, wolf_cap=64)
    assert env.lanes_per_env == lpe
    oracles = [OracleEnv(overrides, seed=seed, env_id=base + i) for i in range(n)]
    rng = np.random.default_rng(lpe)
    obs = env.reset()
    cur = [o.reset() for o in oracles]
    for t in range(steps + 1):
        g, f, r, s = (x.cpu().numpy() for x in obs)
        st = env.export_state()
        for i, o in enumerate(oracles):
            assert np.array_equal(g[i], cur[i][0]) and (int(f[i]), int(r[i]), int(s[i])) == cur[i][1:], (lpe, t, i)
            hs = o.hidden_state()
            assert (st["x"][i], st["y"][i], st["turn"][i]) == (hs["x"], hs["y"], hs["turn"]) and _wolves(st, i) == hs["wolves"]
            assert mask_words_to_int(st["bush_mask"][i]) == window_mask_from_bushes(hs), (lpe, t, i)
        if t == steps:
            break
        acts = np.array([pick_action(rng, cur[i][0], env.n_actions, greedy) for i in range(n)], dtype=np.uint8)
        obs, reward, done, _ = env.step(torch.from_numpy(acts).cuda())
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        for i, o in enumerate(oracles):
            c, rr, d = o.step(int(acts[i]))
            assert np.float32(rr) == reward[i] and d == bool(done[i]), (lpe, t, i)
            cur[i] = o.reset() if d else c
    assert env.stats()["steps"] == n * steps and env.stats()["overflows"] == 0
    env.close()


def test_lanes_per_env_variants_agree_on_a_full_batch(monkeypatch):
    n, steps = 4096, 48
    acts = torch.randint(0, 5, (steps, n), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    ref = None
    for lpe in (1, 4, 8, 16, 32):
        monkeypatch.setenv("WAB_LPE", str(lpe))
        env = _vec(n, seed=12)
        env.reset()
        o, r, d, i = env.step_many(acts)
        got = [x.clone() for x in (o.grids, o.food, o.role, o.status, r, d, i["info"])] + [env.stats()]
        if ref is None:
            ref = got
        else:
            for x, y in zip(ref[:-1], got[:-1]):
                assert torch.equal(x, y), lpe
            assert ref[-1] == got[-1]
        env.close()
    # the thread-per-env kernel built for 7 and 8 resident CTAs per SM (tighter register caps, picked for batches of
    # just over one wave) gives the same answers
    monkeypatch.setenv("WAB_LPE", "1")
    for mb in (7, 8):
        monkeypatch.setenv("WAB_MB", str(mb))
        env = _vec(n, seed=12)
        env.reset()
        o, r, d, i = env.step_many(acts)
        for x, y in zip(ref[:-1], (o.grids, o.food, o.role, o.status, r, d, i["info"])):
            assert torch.equal(x, y), mb
        assert ref[-1] == env.stats()
        env.close()
    monkeypatch.delenv("WAB_MB")
    monkeypatch.delenv("WAB_LPE")
    auto = _vec(n, seed=12)
    assert auto.lanes_per_env in (4, 8, 16)         # a 4096-env batch is spread over several lanes per env
    auto.close()


def test_step_many_equals_repeated_step_and_sharding_is_invisible():
    n, steps = 4096, 64
    acts = torch.randint(0, 5, (steps, n), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    a = _vec(n, seed=3)
    a.reset()
    outs = []
    for t in range(steps):
        o, r, d, i = a.step(acts[t])
        outs.append((o.grids.clone(), o.food.clone(), o.role.clone(), o.status.clone(), r.clone(), d.clone(), i["info"].clone()))
    b = _vec(n, seed=3)
    b.reset()
    o, r, d, i = b.step_many(acts)
    for t in range(steps):
        got = (o.grids[t], o.food[t], o.role[t], o.status[t], r[t], d[t], i["info"][t])
        for x, y in zip(outs[t], got):
            assert torch.equal(x, y), t
    sa, sb = a.export_state(), b.export_state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    # two shards with global ids = one batch
    lo, hi = _vec(1024, seed=3, env_id_base=0), _vec(n - 1024, seed=3, env_id_base=1024)
    lo.reset(), hi.reset()
    ol, rl, dl, _ = lo.step_many(acts[:, :1024].contiguous())
    oh, rh, dh, _ = hi.step_many(acts[:, 1024:].contiguous())
    assert torch.equal(torch.cat([ol.grids, oh.grids], 1), o.grids) and torch.equal(torch.cat([rl, rh], 1), r)
    assert torch.equal(torch.cat([dl, dh], 1), d)
    assert a.stats() == b.stats()
    for e in (a, b, lo, hi):
        e.close()


@pytest.mark.parametrize("lpe", [1, 8, 32])
def test_step_many_on_a_ragged_batch(lpe, monkeypatch):
    """N = 77 is not a multiple of 16: every step's slab starts at a different 16-byte phase."""
    monkeypatch.setenv("WAB_LPE", str(lpe))
    n, steps = 77, 23
    acts = torch.randint(0, 5, (steps, n), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(8))
    a, b = _vec(n, seed=2), _vec(n, seed=2)
    a.reset(), b.reset()
    o, r, d, i = a.step_many(acts)
    canary = torch.full((steps, n, 3, 11, 11), 7, dtype=torch.uint8, device="cuda")
    for t in range(steps):
        ob, rb, db, ib = b.step(acts[t])
        canary[t] = ob.grids
        assert torch.equal(o.grids[t], ob.grids) and torch.equal(r[t], rb) and torch.equal(d[t], db), (lpe, t)
        assert torch.equal(o.food[t], ob.food) and torch.equal(i["info"][t], ib["info"])
    assert int(canary.max()) <= 1
    a.close(), b.close()


def test_full_size_checksum_against_oracle():
    """BASELINE config 2 (4096 default envs): position-weighted checksum of every observation of
    every step equals the CPU oracle's (a checksum of checksums over 4096 x 400 env-steps)."""
    n, steps, seed = 4096, 400, 0
    acts = torch.randint(0, 5, (steps, n), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    env = _vec(n, seed=seed)
    env.reset()
    o, r, d, _ = env.step_many(acts)
    w = torch.arange(1, 364, device="cuda", dtype=torch.int64)
    cs = (o.grids.view(steps, n, 363).long() * w).sum() + 1000 * o.food.long().sum() + 100000 * o.role.long().sum() \
        + 200000 * o.status.long().sum() + 400000 * d.long().sum()
    n_steps, want = wab_oracle.run(None, seed, n, steps, acts.cpu().numpy())
    assert n_steps == n * steps and int(cs.item()) == want
    # size-independent invariants
    assert int(o.grids[:, :, 2, 5, 5].min()) == 1 and int(o.grids[:, :, 2].sum()) == n * steps
    assert int(o.status.max()) == 0                      # auto-reset: returned obs is always a live ostrich
    st = env.stats()
    assert st["episodes"] == int(d.sum()) and st["steps"] == n * steps
    env.close()


def test_million_env_checksum_against_oracle():
    """BASELINE's largest v1 batch: 1,048,576 envs x 12 lockstep steps (12.6 M env-steps, thread-per-env kernel, every
    observation byte of every step) against the CPU oracle's checksum of the same run."""
    n, steps, seed = 1 << 20, 12, 3
    acts = torch.randint(0, 5, (steps, n), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(8))
    env = _vec(n, seed=seed)
    assert env.lanes_per_env == 1
    env.reset()
    o, r, d, _ = env.step_many(acts)
    w = torch.arange(1, 364, device="cuda", dtype=torch.int64)
    cs = 0
    for t in range(steps):                                  # per step: keeps the int64 temporaries at 3 GB
        cs += int((o.grids[t].view(n, 363).long() * w).sum().item())
    cs += int((1000 * o.food.long().sum() + 100000 * o.role.long().sum() + 200000 * o.status.long().sum()
               + 400000 * d.long().sum()).item())
    n_steps, want = wab_oracle.run(None, seed, n, steps, acts.cpu().numpy())
    assert n_steps == n * steps and cs == want
    st = env.stats()
    assert st["steps"] == n * steps and st["overflows"] == 0 and st["episodes"] == int(d.sum())
    env.close()


@pytest.mark.parametrize("mapped", ["0", "1"])
def test_host_buffer_path_and_masked_reset(mapped, monkeypatch):
    """Host entry points: staged copies (0) and the thread-per-env kernel writing the pinned block directly (1, the
    default for small batches) — both equal to the device path."""
    monkeypatch.setenv("WAB_HOST_MAPPED", mapped)
    n = 300
    a, b = _vec(n, seed=9), _vec(n, seed=9)
    hb = a.alloc_host_buffers(pinned=True)
    a.reset_host(hb)
    ob = b.reset()
    assert np.array_equal(hb["grids"].numpy(), ob.grids.cpu().numpy())
    rng = np.random.default_rng(2)
    for t in range(40):
        acts = rng.integers(0, 5, n).astype(np.uint8)
        hb["actions"].copy_(torch.from_numpy(acts))
        a.step_host(hb)
        o, r, d, i = b.step(torch.from_numpy(acts).cuda())
        assert np.array_equal(hb["grids"].numpy(), o.grids.cpu().numpy()) and np.array_equal(hb["reward"].numpy(), r.cpu().numpy())
        assert np.array_equal(hb["done"].numpy().astype(bool), d.cpu().numpy()) and np.array_equal(hb["food"].numpy(), o.food.cpu().numpy())
    # the seven-pointer entry point (no packed block) gives the same answers
    loose = {k: v.clone() for k, v in hb.items() if isinstance(v, torch.Tensor) and k != "block"}
    acts = rng.integers(0, 5, n).astype(np.uint8)
    loose["actions"].copy_(torch.from_numpy(acts))
    a.step_host(loose)
    o, r, d, i = b.step(torch.from_numpy(acts).cuda())
    assert np.array_equal(loose["grids"].numpy(), o.grids.cpu().numpy()) and np.array_equal(loose["reward"].numpy(), r.cpu().numpy())
    # buffers handed back (the library forgets its cached aliases / graph for their addresses), fresh ones — at an odd
    # offset inside a pinned allocation, so the block is NOT 16-byte aligned and the mapped path must stand down — work too
    from wab_gym_b200 import _lib
    a.free_host_buffers(hb)
    assert not hb
    hb2 = a.alloc_host_buffers(pinned=True)
    odd = torch.empty(hb2["block"].numel() + 64, dtype=torch.uint8).pin_memory()
    for blk in (hb2["block"], odd[4:4 + hb2["block"].numel()]):
        acts = rng.integers(0, 5, n).astype(np.uint8)
        hb2["actions"].copy_(torch.from_numpy(acts))
        _lib.check(a.lib.wab_vec_step_host_packed(a._h, hb2["actions"].data_ptr(), blk.data_ptr(), a._stream()))
        o, r, d, i = b.step(torch.from_numpy(acts).cuda())
        assert np.array_equal(blk[:o.grids.numel()].numpy().reshape(o.grids.shape), o.grids.cpu().numpy())
    # masked reset: only the selected envs start a new episode
    before = b.export_state()
    prev = [t.cpu().numpy().copy() for t in o]
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[::3] = 1
    again = [t.cpu().numpy() for t in b.reset(mask)]
    after = b.export_state()
    sel = mask.cpu().numpy().astype(bool)
    for was, now in zip(prev, again):         # the others get their last observation again (bush just eaten included)
        assert np.array_equal(was[~sel], now[~sel])
    assert np.array_equal(after["episode"][sel], before["episode"][sel] + 1) and np.all(after["turn"][sel] == 0)
    assert np.array_equal(after["episode"][~sel], before["episode"][~sel]) and np.array_equal(after["x"][~sel], before["x"][~sel])
    a.close(), b.close()


def test_bad_actions_are_counted_not_dropped():
    env = _vec(64, seed=1)
    env.reset()
    acts = torch.full((64,), 9, dtype=torch.uint8, device="cuda")
    _, _, _, info = env.step(acts)
    assert int(((info["info"] >> 3) & 1).sum()) == 64 and env.stats()["bad_actions"] == 64
    env.close()


def test_unaligned_or_missing_buffers_are_rejected():
    from wab_gym_b200 import _lib
    env = _vec(32)
    L = env.lib
    obs = env._obs_struct(env._out)
    assert L.wab_vec_step(env._h, None, obs, None, None, None, None) == 1
    bad = _lib.WabObs(env._out["grids"].data_ptr() + 1, env._out["food"].data_ptr(), env._out["role"].data_ptr(),
                      env._out["status"].data_ptr())
    assert L.wab_vec_reset(env._h, None, bad, None) == 2
    env.close()


def _ref_features(grids, food, role, status):
    """PragmaticObsWrapper features through the host build of the same header (itself pinned to the
    reference's known-answer tests and wrapper in tests/test_features.py)."""
    from tests import hostsim
    return hostsim.features(grids[0], grids[1], food, role, status)


@pytest.mark.parametrize("name", ["defaults", "restrict_view", "dense"])
def test_fused_and_standalone_features(name):
    overrides, greedy = OPTION_SETS[name]
    n, steps = 130, 60
    env = _vec(n, overrides, seed=21, features=True, wolf_cap=64)
    rng = np.random.default_rng(6)
    obs = env.reset()
    feats = env.last_features
    for t in range(steps):
        g, f, r, s = (x.cpu().numpy() for x in obs)
        fused = feats.cpu().numpy()
        alone = env.pragmatic_features(obs).cpu().numpy()
        assert np.array_equal(fused, alone), t
        for i in range(0, n, 7):
            assert np.array_equal(fused[i], _ref_features(g[i], int(f[i]), int(r[i]), int(s[i]))), (t, i)
        flat = env.flatten_features(feats).cpu().numpy()
        assert flat.shape == (n, env.flat_dim) and env.flat_dim == 408 + int(env.game_options["turns_to_empty_food"]) + 1
        i = int(rng.integers(0, n))
        want = []
        for k in range(24):
            oh = np.zeros(12 if (k % 12) < 8 else 11, np.float32); oh[fused[i][k]] = 1; want.append(oh)
        for k, dim in ((24, 2), (25, env.flat_dim - 408), (26, 2), (27, 3)):
            oh = np.zeros(dim, np.float32); oh[fused[i][k]] = 1; want.append(oh)
        from wab_gym_b200.config import GATHERER_TILE_MASK, LOOKOUT_TILE_MASK
        vm = np.zeros(121, np.float32)
        if env.game_options["restrict_view"]:
            vm = (GATHERER_TILE_MASK if r[i] == 1 else LOOKOUT_TILE_MASK).reshape(-1).astype(np.float32)
        want.append(vm)
        assert np.array_equal(flat[i], np.concatenate(want)), (t, i)
        if t % 40 == 0:                                   # the fused policy-input kernel: flatten + noise + cast
            ctr = torch.full((1,), 5 + t, dtype=torch.int64, device="cuda")
            for dt in (torch.float32, torch.bfloat16):
                buf = torch.empty(n, env.flat_dim, dtype=dt, device="cuda")
                assert np.array_equal(env.flatten_features_noisy(feats, buf, 0.0, ctr).float().cpu().numpy(), flat)
            a1 = env.flatten_features_noisy(feats, torch.empty(n, env.flat_dim, device="cuda"), 0.01, ctr).cpu().numpy()
            a2 = env.flatten_features_noisy(feats, torch.empty(n, env.flat_dim, device="cuda"), 0.01, ctr).cpu().numpy()
            ctr += 1
            a3 = env.flatten_features_noisy(feats, torch.empty(n, env.flat_dim, device="cuda"), 0.01, ctr).cpu().numpy()
            noise = a1 - flat
            assert np.array_equal(a1, a2) and not np.array_equal(a1, a3)
            assert noise.min() >= 0.0 and noise.max() < 0.01 + 1e-6 and abs(float(noise.mean()) - 0.005) < 2e-4
        acts = np.array([pick_action(rng, g[j], env.n_actions, greedy) for j in range(n)], dtype=np.uint8)
        obs, _, _, info = env.step(torch.from_numpy(acts).cuda())
        feats = info["features"]
    env.close()


def test_actor_critic_rollout_runs_on_device():
    """BASELINE config 5 in miniature: policy consumes device-resident observations; graph replay and
    eager stepping give the same episode statistics for the same seeds."""
    from wab_gym_b200.policy import Policy, Rollout
    torch.manual_seed(0)
    env = _vec(512, seed=4, features=True)
    pol = Policy(env.flat_dim, env.n_actions)
    assert env.flat_dim == 449 and sum(p.numel() for p in pol.parameters()) == 449 * 128 + 128 + 128 * 150 + 150 + 150 * 128 + 128 + 128 * 5 + 5 + 128 + 1
    ro = Rollout(env, pol, use_graph=False)
    ro.run(50)
    st = env.stats()
    assert st["steps"] == 512 * 50 and st["bad_actions"] == 0 and st["episodes"] > 0
    probs, value = ro.policy(ro.flat)
    assert torch.allclose(probs.sum(-1), torch.ones(512, device="cuda"), atol=1e-5) and value.shape == (512, 1)
    env.close()
    env2 = _vec(512, seed=4, features=True)
    rg = Rollout(env2, pol, use_graph=True)
    rg.run(20)
    assert env2.stats()["steps"] >= 512 * 20 and env2.stats()["bad_actions"] == 0
    env2.close()


def test_device_categorical_sampler_follows_the_probabilities():
    env = _vec(64, seed=1)
    n = 1 << 20
    p = torch.tensor([0.1, 0.2, 0.3, 0.25, 0.15], device="cuda")
    ctr = torch.zeros(1, dtype=torch.int64, device="cuda")
    for dt, tol in ((torch.float32, 2e-3), (torch.bfloat16, 6e-3)):
        probs = p.to(dt).expand(n, 5).contiguous()
        a = env.sample_actions(probs, torch.empty(n, dtype=torch.uint8, device="cuda"), ctr, seed=7)
        freq = torch.bincount(a.long(), minlength=5).float() / n
        want = probs[0].float() / probs[0].float().sum()
        assert int(a.max()) <= 4 and float((freq - want).abs().max()) < tol, (dt, freq)
        again = env.sample_actions(probs, torch.empty(n, dtype=torch.uint8, device="cuda"), ctr, seed=7)
        assert torch.equal(a, again)                        # keyed: same counter, same draws
        ctr += 1
        assert not torch.equal(a, env.sample_actions(probs, torch.empty(n, dtype=torch.uint8, device="cuda"), ctr, seed=7))
    onehot = torch.eye(5, device="cuda")[torch.arange(n, device="cuda") % 5].contiguous()
    a = env.sample_actions(onehot, torch.empty(n, dtype=torch.uint8, device="cuda"), ctr)
    assert torch.equal(a.long(), torch.arange(n, device="cuda") % 5)
    env.close()


def test_batched_a2c_update_trains_on_device():
    """SURVEY 8f-2: the reference's finish_episode (actor_critic.py:128-169) batched over envs."""
    from wab_gym_b200.a2c import A2CTrainer
    torch.manual_seed(1)
    env = _vec(1024, seed=8, features=True)
    tr = A2CTrainer(env, horizon=40, lr=1e-3)
    before = [p.detach().clone() for p in tr.policy.parameters()]
    out = [tr.train_iteration() for _ in range(3)]
    assert all(torch.isfinite(o["loss"]).item() for o in out)
    assert any(not torch.equal(a, b.detach()) for a, b in zip(before, tr.policy.parameters()))
    assert env.stats()["steps"] == 1024 * 40 * 3 and env.stats()["bad_actions"] == 0
    env.close()


@pytest.mark.parametrize("lpe", [1, 16])
@pytest.mark.parametrize("n", [33, 4096])
def test_outputs_never_touch_guard_bytes(lpe, n, monkeypatch):
    """compute-sanitizer is closed on this pool, so bounds are checked with canaries: every output lives inside a
    larger buffer whose 256 guard bytes on either side must survive reset / step / step_many untouched."""
    monkeypatch.setenv("WAB_LPE", str(lpe))
    steps, G = 9, 256
    env = _vec(n, seed=5, features=True, game_options={"chance_wolf_on_square": 0.01})

    def guarded(shape, dtype):
        numel = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        raw = torch.full((numel + 2 * G,), 0xAB, dtype=torch.uint8, device="cuda")
        return raw, raw[G:G + numel].view(dtype).view(shape)

    shapes = {"grids": ((steps, n, 3, 11, 11), torch.uint8), "food": ((steps, n), torch.uint8), "role": ((steps, n), torch.uint8),
              "status": ((steps, n), torch.uint8), "reward": ((steps, n), torch.float32), "done": ((steps, n), torch.uint8),
              "info": ((steps, n), torch.uint8), "features": ((steps, n, 28), torch.uint8)}
    raws, out = {}, {}
    for k, (shape, dt) in shapes.items():
        raws[k], out[k] = guarded(shape, dt)
    env.reset()
    acts = torch.randint(0, 5, (steps, n), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(2))
    env.step_many(acts, out=out)
    torch.cuda.synchronize()
    for k, raw in raws.items():
        assert int((raw[:G] != 0xAB).sum()) == 0 and int((raw[-G:] != 0xAB).sum()) == 0, (k, lpe, n)
    assert int(out["grids"].max()) <= 1 and int(out["features"].max()) <= 40 and int(out["status"].max()) == 0
    env.close()


@pytest.mark.parametrize("name", ["defaults", "six_actions_random_start", "dense"])
def test_batch_without_auto_reset_keeps_reporting_done(name):
    """VecEnv(auto_reset=False): the reference's behaviour after an episode ends (wab_env.py:328-340 — done is
    returned again, the dead ostrich still moves, reveals bushes and can starve after being killed), for a batch;
    fp64 food, masked reset of the finished envs every few steps."""
    overrides, greedy = OPTION_SETS[name]
    n, steps, seed = 48, 220, 13
    env = _vec(n, overrides, seed=seed, auto_reset=False, wolf_cap=64)
    assert env.game.food_mode == 0
    oracles = [OracleEnv(overrides, seed=seed, env_id=i) for i in range(n)]
    rng = np.random.default_rng(3)
    obs = env.reset()
    cur = [o.reset() for o in oracles]
    done_now = np.zeros(n, bool)
    for t in range(steps):
        g, f, r, s = (x.cpu().numpy() for x in obs)
        for i in range(n):
            assert np.array_equal(g[i], cur[i][0]) and (int(f[i]), int(r[i]), int(s[i])) == cur[i][1:], (t, i)
        if t % 7 == 6 and done_now.any():                       # reset only the envs that are done
            mask = torch.from_numpy(done_now.astype(np.uint8)).cuda()
            obs = env.reset(mask)
            for i in np.nonzero(done_now)[0]:
                cur[i] = oracles[i].reset()
            done_now[:] = False
            continue
        acts = np.array([pick_action(rng, cur[i][0], env.n_actions, greedy) for i in range(n)], dtype=np.uint8)
        obs, reward, done, _ = env.step(torch.from_numpy(acts).cuda())
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        for i, o in enumerate(oracles):
            cur[i], rr, d = o.step(int(acts[i]))
            assert np.float32(rr) == reward[i] and d == bool(done[i]), (t, i)
            done_now[i] = d
    st = env.export_state()
    for i, o in enumerate(oracles):
        hs = o.hidden_state()
        assert st["food"][i] == hs["food"] and (st["x"][i], st["y"][i], st["status"][i]) == (hs["x"], hs["y"], hs["status"])
    env.close()


@pytest.mark.parametrize("case", range(12))
def test_random_option_sets_match_oracle_on_device(case):
    """Randomised game options (tests/test_fuzz_options.random_options): 96 lockstep envs x 160 steps per case, the
    CUDA path against one oracle env per env (observations, reward, done every step) and, over 2,048 envs x 96 steps,
    against the oracle's batch checksum."""
    from tests.test_fuzz_options import random_options
    rng = np.random.default_rng(1000 + case)
    opts = random_options(rng)
    n, steps, seed = 96, 160, 40 + case
    env = _vec(n, opts, seed=seed, wolf_cap=64, force_f64_food=bool(case & 1))
    oracles = [OracleEnv(opts, seed=seed, env_id=i) for i in range(n)]
    obs = env.reset()
    cur = [o.reset() for o in oracles]
    for t in range(steps):
        g, f, r, s = (x.cpu().numpy() for x in obs)
        for i in range(n):
            assert np.array_equal(g[i], cur[i][0]) and (int(f[i]), int(r[i]), int(s[i])) == cur[i][1:], (case, t, i, opts)
        acts = rng.integers(0, env.n_actions, n).astype(np.uint8)
        obs, reward, done, _ = env.step(torch.from_numpy(acts).cuda())
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        for i, o in enumerate(oracles):
            cur[i], rr, d = o.step(int(acts[i]))
            assert np.float32(rr) == reward[i] and d == bool(done[i]), (case, t, i, opts)
            if d:
                cur[i] = o.reset()
    assert env.stats()["overflows"] == 0
    env.close()
    # batch checksum at a larger size (thread-per-env and lanes-per-env kernels alike)
    n2, steps2 = 2048, 96
    big = _vec(n2, opts, seed=seed, wolf_cap=64)
    acts = torch.randint(0, big.n_actions, (steps2, n2), dtype=torch.uint8, device="cuda",
                         generator=torch.Generator("cuda").manual_seed(case))
    big.reset()
    o, r, d, _ = big.step_many(acts)
    w = torch.arange(1, 364, device="cuda", dtype=torch.int64)
    cs = (o.grids.view(steps2, n2, 363).long() * w).sum() + 1000 * o.food.long().sum() + 100000 * o.role.long().sum() \
        + 200000 * o.status.long().sum() + 400000 * d.long().sum()
    n_steps, want = wab_oracle.run(opts, seed, n2, steps2, acts.cpu().numpy())
    assert big.stats()["overflows"] == 0                 # 64 wolf slots: no fuzzed option set gets near
    assert n_steps == n2 * steps2 and int(cs.item()) == want, (case, opts)
    big.close()


@pytest.mark.parametrize("lpe", [1, 8])
def test_wolf_packs_beyond_32_stay_exact_on_device(lpe, monkeypatch):
    """The reference's wolf list is unbounded (wab_env.py:570-575). ~24 wolves alive per env with peaks above 32 (64
    slots): observations, reward, done and the wolf multiset stay equal to the oracle, and nothing overflows."""
    monkeypatch.setenv("WAB_LPE", str(lpe))
    opts = {"chance_wolf_on_square": 0.05, "god_mode": True, "max_turns": 400, "turns_to_empty_food": 200, "starting_food": 1.0}
    n, steps, seed = 24, 300, 11
    env = _vec(n, opts, seed=seed, wolf_cap=64)
    oracles = [OracleEnv(opts, seed=seed, env_id=i) for i in range(n)]
    rng = np.random.default_rng(5)
    obs = env.reset()
    cur = [o.reset() for o in oracles]
    peak = 0
    for t in range(steps):
        g, f, r, s = (x.cpu().numpy() for x in obs)
        for i in range(n):
            assert np.array_equal(g[i], cur[i][0]) and (int(f[i]), int(r[i]), int(s[i])) == cur[i][1:], (t, i)
        if t % 25 == 24:
            st = env.export_state()
            for i, o in enumerate(oracles):
                assert _wolves(st, i) == o.hidden_state()["wolves"], (t, i)
                peak = max(peak, int(st["n_wolves"][i]))
        acts = rng.integers(0, 5, n).astype(np.uint8)
        obs, reward, done, _ = env.step(torch.from_numpy(acts).cuda())
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        for i, o in enumerate(oracles):
            c, rr, d = o.step(int(acts[i]))
            assert np.float32(rr) == reward[i] and d == bool(done[i]), (t, i)
            cur[i] = o.reset() if d else c
    assert peak > 32 and env.stats()["overflows"] == 0
    env.close()


@pytest.mark.parametrize("lpe", [4, 8, 16, 32])
@pytest.mark.parametrize("name", ["defaults", "dense", "six_actions_random_start", "restrict_view", "tiny_bushes"])
def test_two_warp_pipeline_equals_single_steps(lpe, name, monkeypatch):
    """Multi-step launches of the lanes-per-env geometries run as a pair of warps per env group: one runs the rules and
    parks each step's planes and scalars in a ring of shared-memory slots, the other publishes them (wab_step_pipe_kernel).
    Every output of launches of 4, 5, 23, 64 and 131 steps on a ragged batch — observations, features, reward, done, info,
    the position history, the hidden state and the statistics — equals what single-step launches give, and so does the
    same launch with the pipeline switched off."""
    monkeypatch.setenv("WAB_LPE", str(lpe))
    monkeypatch.setenv("WAB_PIPE", "2")             # always (the default uses it only while the batch leaves issue slots free)
    overrides, _ = OPTION_SETS[name]
    n, seed = 45, 321
    a = _vec(n, overrides, seed=seed, features=True, wolf_cap=64, ego=True)
    b = _vec(n, overrides, seed=seed, features=True, wolf_cap=64, ego=True)
    c = _vec(n, overrides, seed=seed, features=True, wolf_cap=64, ego=True)
    assert a.lanes_per_env == lpe
    gen = torch.Generator(device="cuda").manual_seed(100 + lpe)
    a.reset(); b.reset(); c.reset()
    for T in (4, 5, 23, 64, 131):
        acts = torch.randint(0, a.n_actions, (T, n), dtype=torch.uint8, device="cuda", generator=gen)
        acts[T // 2, 3] = 77                                   # a bad action in the middle of the launch
        oa, ra, da, ia = a.step_many(acts)
        monkeypatch.setenv("WAB_PIPE", "0")
        oc, rc, dc, ic = c.step_many(acts)
        monkeypatch.setenv("WAB_PIPE", "2")
        for x, y in zip(oa, oc):
            assert torch.equal(x, y), (lpe, name, T)
        assert torch.equal(ra, rc) and torch.equal(da, dc) and torch.equal(ia["info"], ic["info"])
        assert torch.equal(ia["features"], ic["features"])
        for t in range(T):
            ob, rb, db, ib = b.step(acts[t])
            for x, y in zip(oa, ob):
                assert torch.equal(x[t], y), (lpe, name, T, t)
            assert torch.equal(ra[t], rb) and torch.equal(da[t], db) and torch.equal(ia["info"][t], ib["info"]), (lpe, name, T, t)
            assert torch.equal(ia["features"][t], ib["features"]), (lpe, name, T, t)
        assert torch.equal(a.ego_proximities(), b.ego_proximities()), (lpe, name, T)
        sa, sb, sc = a.export_state(), b.export_state(), c.export_state()
        for k in sa:
            assert np.array_equal(sa[k], sb[k]) and np.array_equal(sa[k], sc[k]), (lpe, name, T, k)
    assert a.stats() == b.stats() == c.stats() and a.stats()["bad_actions"] == 5
    a.close(); b.close(); c.close()


@pytest.mark.parametrize("lpe", [1, 8, 32])
def test_features_only_stepping_equals_full_stepping(lpe, monkeypatch):
    """VecEnv(emit_grids=False): the kernels get d_grids = NULL and never materialise the one-hot grids; the 28 feature
    bytes, scalars, reward, done, info, the statistics and the hidden state equal those of a batch that writes them —
    single-step launches, multi-step launches (pipeline kernel included) and resets."""
    monkeypatch.setenv("WAB_LPE", str(lpe))
    n, seed = 77, 5
    full = _vec(n, OPTION_SETS["dense"][0], seed=seed, features=True, wolf_cap=64)
    lean = _vec(n, OPTION_SETS["dense"][0], seed=seed, features=True, wolf_cap=64, emit_grids=False)
    of, ol = full.reset(), lean.reset()
    assert ol.grids is None and torch.equal(full.last_features, lean.last_features)
    for x, y in zip(of[1:], ol[1:]):
        assert torch.equal(x, y)
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(30):
        a = torch.randint(0, full.n_actions, (n,), dtype=torch.uint8, device="cuda", generator=gen)
        (of, rf, df, jf), (ol, rl, dl, jl) = full.step(a), lean.step(a)
        assert torch.equal(jf["features"], jl["features"]) and torch.equal(rf, rl) and torch.equal(df, dl) and torch.equal(jf["info"], jl["info"])
        assert torch.equal(of.food, ol.food) and torch.equal(of.role, ol.role) and torch.equal(of.status, ol.status)
    for T in (3, 24):
        acts = torch.randint(0, full.n_actions, (T, n), dtype=torch.uint8, device="cuda", generator=gen)
        (of, rf, df, jf), (ol, rl, dl, jl) = full.step_many(acts), lean.step_many(acts)
        assert ol.grids is None
        assert torch.equal(jf["features"], jl["features"]) and torch.equal(rf, rl) and torch.equal(df, dl) and torch.equal(jf["info"], jl["info"])
    sf, sl = full.export_state(), lean.export_state()
    for k in sf:
        assert np.array_equal(sf[k], sl[k]), k
    assert full.stats() == lean.stats()
    with pytest.raises(ValueError):
        _vec(8, seed=1, emit_grids=False)               # no feature buffer to write instead
    full.close(); lean.close()
