"""Replicated handles on the B200: every block of ``VecEnv(P n, replicas=P)``, driven by its own actions, equals a
standalone ``VecEnv(n, env_id_base=base)`` byte for byte, in every kernel family; equal actions give equal blocks; saved
state round-trips through slots; and every refusal of a handle whose env ids repeat comes before any device work."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

P, n, BASE, STEPS = 3, 200, 1000, 300


def _outputs(env, obs, reward, done, info):
    out = [obs.food, obs.role, obs.status, reward, done, info["info"]]
    if obs.grids is not None:
        out.append(obs.grids)
    if env.with_features:
        out.append(env.last_features)
    return out


@pytest.mark.parametrize("kind", ["default", "generic", "features_only"])
def test_each_block_equals_a_standalone_env(kind):
    from wab_gym_b200 import VecEnv
    opts = {"width": 13, "height": 13} if kind == "generic" else None
    kw = dict(features=kind != "generic", emit_grids=kind != "features_only")
    rep = VecEnv(P * n, game_options=opts, seed=7, env_id_base=BASE, replicas=P, **kw)
    alone = [VecEnv(n, game_options=opts, seed=7, env_id_base=BASE, **kw) for _ in range(P)]
    assert rep.replicas == P and rep.generic_kernels == (kind == "generic") and rep.game_options["wolves"]
    rep.reset()
    for a in alone:
        a.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(STEPS):
        acts = torch.randint(0, rep.n_actions, (P * n,), generator=gen, device="cuda", dtype=torch.int64).to(torch.uint8)
        got = _outputs(rep, *rep.step(acts))
        for p, a in enumerate(alone):
            want = _outputs(a, *a.step(acts[p * n:(p + 1) * n]))
            for g, w in zip(got, want):
                assert torch.equal(g[p * n:(p + 1) * n], w), (kind, t, p)
    # the blocks really played different episodes (different action streams)
    assert not torch.equal(rep.last_features[:n] if rep.with_features else rep._out["grids"][:n],
                           rep.last_features[n:2 * n] if rep.with_features else rep._out["grids"][n:2 * n])
    st = rep.stats()
    assert st["steps"] == P * n * STEPS and st["killed"] > 0
    for env in [rep] + alone:
        env.close()


def test_equal_actions_give_equal_blocks():
    from wab_gym_b200 import VecEnv
    rep = VecEnv(P * n, seed=11, env_id_base=BASE, replicas=P, features=True)
    rep.reset()
    gen = torch.Generator(device="cuda").manual_seed(5)
    for _ in range(120):
        acts = torch.randint(0, rep.n_actions, (n,), generator=gen, device="cuda").to(torch.uint8).repeat(P)
        out = _outputs(rep, *rep.step(acts))
        for x in out:
            blocks = x.view(P, n, *x.shape[1:])
            for p in range(1, P):
                assert torch.equal(blocks[p], blocks[0])
    rep.close()


def test_save_and_load_through_slots_round_trips():
    from wab_gym_b200 import VecEnv
    rep = VecEnv(P * n, seed=4, env_id_base=BASE, replicas=P, features=True)
    rep.reset()
    gen = torch.Generator(device="cuda").manual_seed(8)
    acts = [torch.randint(0, rep.n_actions, (P * n,), generator=gen, device="cuda").to(torch.uint8) for _ in range(60)]
    for a in acts[:20]:
        rep.step(a)
    st = rep.save_state()
    assert torch.equal(st.env_ids, (torch.arange(P * n) % n) + BASE)
    first = [[x.clone() for x in _outputs(rep, *rep.step(a))] for a in acts[20:]]
    rep.load_state(st, slots=torch.arange(P * n))
    for a, want in zip(acts[20:], first):
        for g, w in zip(_outputs(rep, *rep.step(a)), want):
            assert torch.equal(g, w)
    # a record moves between blocks: block 2's env j loaded into block 0 continues as block 2's env j
    part = rep.save_state(torch.arange(2 * n, 3 * n))
    rep.load_state(part, slots=torch.arange(0, n))
    for a in acts[:30]:
        a = a.clone()
        a[:n] = a[2 * n:]
        for x in _outputs(rep, *rep.step(a)):
            assert torch.equal(x[:n], x[2 * n:])
    rep.close()


def test_refusals_come_before_any_device_work():
    from wab_gym_b200 import VecEnv, PPOPopulation
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.ppo import PPOTrainer
    with pytest.raises(ValueError, match="replicas"):
        VecEnv(300, replicas=7)
    with pytest.raises(ValueError, match="replicas"):
        VecEnv(300, replicas=0)
    env = VecEnv(4 * 128, seed=1, replicas=4, features=True)
    st = env.save_state()
    for call in (env.state_dict, lambda: env.load_state_dict({}), lambda: env.load_state(st),
                 lambda: A2CTrainer(env, tensor_cores=True), lambda: PPOTrainer(env), lambda: PPOPopulation(env, 4)):
        with pytest.raises(ValueError, match="replicas"):
            call()
    # nothing above reset or loaded the handle: the replica layout can still be set, and the envs were never stepped
    assert env.lib.wab_vec_set_replicas(env._h, 2) == 0
    assert env.stats()["steps"] == 0
    env.reset()
    assert env.lib.wab_vec_set_replicas(env._h, 2) == 2                 # WAB_E_CONFIG after the first reset
    fresh = VecEnv(300, seed=1)
    assert fresh.lib.wab_vec_set_replicas(fresh._h, 7) == 2             # does not divide n_envs
    assert fresh.lib.wab_vec_set_replicas(fresh._h, 0) == 2
    assert fresh.lib.wab_vec_set_replicas(None, 3) == 1
    assert fresh.lib.wab_vec_set_replicas(fresh._h, 1) == 0             # one replica: the unreplicated handle
    fresh.reset()
    assert torch.equal(fresh.save_state().env_ids, torch.arange(300))
    env.close()
    fresh.close()
