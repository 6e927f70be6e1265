"""Populations on the B200: the population forward and PPO backward against P single-policy calls, ``PPOPopulation``
against P standalone ``PPOTrainer`` runs, resume and member state, and the ABI's refusals. Every comparison is bit for
bit."""
import copy
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

P, n, T = 3, 256, 16
GUARD = 4096


def _env(num_envs, base=0, seed=5):
    from wab_gym_b200 import VecEnv
    return VecEnv(num_envs, seed=seed, env_id_base=base, features=True)


def _policies(env, seed=1):
    """P different reference networks, scaled so both leaky branches and the upper clamp are populated."""
    from wab_gym_b200.policy import Policy
    out = []
    for p in range(P):
        torch.manual_seed(seed + 17 * p)
        pol = Policy(env.flat_dim, env.n_actions).cuda()
        with torch.no_grad():
            for lin in (pol.affine1, pol.affine2, pol.affine3):
                lin.weight.mul_(3.0)
            pol.affine3.bias[:32] += 3.5
            pol.action_head.weight.mul_(4.0)
        out.append(pol)
    return out


def _guarded(shape, fill, dtype=torch.float32):
    """A tensor of `shape` inside a buffer whose GUARD elements on each side hold `fill`; returns (view, check)."""
    numel = 1
    for s in shape:
        numel *= s
    buf = torch.full((numel + 2 * GUARD,), fill, dtype=dtype, device="cuda")
    view = buf[GUARD:GUARD + numel].view(*shape)
    return view, lambda: bool((buf[:GUARD] == fill).all()) and bool((buf[-GUARD:] == fill).all())


@pytest.mark.parametrize("noise", [0.01, 0.0])
def test_forward_equals_standalone_forward_per_member(noise):
    from wab_gym_b200.policy import PolicyPopulationTC, PolicyTrainTC
    env = _env(P * n)
    env.reset()
    pols = _policies(env)
    pop = PolicyPopulationTC(env, pols)
    feats = env.last_features.clone()
    ctr = torch.full((1,), 9, dtype=torch.int64, device="cuda")
    A = env.n_actions
    acts, ok_a = _guarded((P * n,), 250, torch.uint8)
    value, ok_v = _guarded((P * n,), -777.0)
    probs, ok_p = _guarded((P * n, A), -777.0)
    logp, ok_l = _guarded((P * n,), -777.0)
    z3, ok_z = _guarded((P * n, 128), -777.0)
    pop.forward_sample(feats, acts, value=value, probs=probs, logp=logp, noise_scale=noise, counter=ctr, seed=17, z3=z3)
    assert ok_a() and ok_v() and ok_p() and ok_l() and ok_z()
    for p in range(P):
        sl = slice(p * n, (p + 1) * n)
        env_p = _env(n, base=p * n)
        tc = PolicyTrainTC(env_p, pols[p])
        a, v, pr, lp, z = (torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, device="cuda"),
                           torch.empty(n, A, device="cuda"), torch.empty(n, device="cuda"), torch.empty(n, 128, device="cuda"))
        tc.forward_sample(feats[sl].contiguous(), tc.heads, a, value=v, probs=pr, logp=lp, noise_scale=noise, counter=ctr,
                          seed=17, z3=z)
        assert torch.equal(acts[sl], a) and torch.equal(value[sl], v) and torch.equal(probs[sl], pr)
        assert torch.equal(logp[sl], lp) and torch.equal(z3[sl], z)
        env_p.close()
    # members really differ: the same features under member 0's weights give other outputs
    assert not torch.equal(value[:n], value[n:2 * n])
    env.close()


def _rollout(env, pop, noise=0.01):
    N = env.num_envs
    feats = torch.empty(T, N, 28, dtype=torch.uint8, device="cuda")
    ctrs = torch.empty(T, dtype=torch.int64, device="cuda")
    acts = torch.empty(T, N, dtype=torch.uint8, device="cuda")
    lp = torch.empty(T, N, device="cuda")
    ctr = torch.full((1,), 100, dtype=torch.int64, device="cuda")
    for t in range(T):
        ctr += 1
        feats[t].copy_(env.last_features)
        ctrs[t:t + 1].copy_(ctr)
        pop.forward_sample(feats[t], acts[t], logp=lp[t], noise_scale=noise, counter=ctr, seed=17)
        env.step(acts[t])
    return feats, ctrs, acts, lp


def test_backward_equals_standalone_backward_per_member():
    from wab_gym_b200.policy import PolicyPopulationTC, PolicyTrainTC
    env = _env(P * n)
    env.reset()
    pols = _policies(env, seed=3)
    pop = PolicyPopulationTC(env, pols)
    feats, ctrs, acts, lp = _rollout(env, pop)
    N, TN = P * n, T * n
    g = torch.Generator(device="cuda").manual_seed(11)
    adv = torch.randn(T, N, device="cuda", generator=g)
    target = torch.randn(T, N, device="cuda", generator=g)
    logp_old = (lp + 0.5 * torch.randn(T, N, device="cuda", generator=g)).contiguous()
    clips = [0.1, 0.2, 0.3]
    ratio = torch.exp(lp - logp_old)
    for p in range(P):                                       # >= 5 % of each member's rows on each clip side
        sl = slice(p * n, (p + 1) * n)
        r, a = ratio[:, sl], adv[:, sl]
        assert float(((a > 0) & (r > 1 + clips[p])).float().mean()) >= 0.05
        assert float(((a < 0) & (r < 1 - clips[p])).float().mean()) >= 0.05
    counts = [TN - 1, TN - 300, TN // 2 + 5]                 # ragged, below T n
    M = max(counts) + 9
    rows = torch.full((P, M), -5, dtype=torch.int32)         # entries past a member's count are never read
    local = torch.full((P, M), -5, dtype=torch.int32)        # the standalone lists: a dropped entry is an invalid row
    for p in range(P):
        perm = torch.randperm(TN, generator=torch.Generator().manual_seed(p)).to(torch.int32)[:counts[p]]
        glob = (perm // n) * N + p * n + perm % n
        loc = perm.clone()
        glob[7], loc[7] = glob[3], loc[3]                    # a repeated entry counts twice
        glob[20], loc[20] = T * N + 3, -1                    # outside [0, T N)
        other = (p + 1) % P                                  # another member's row
        glob[41], loc[41] = 2 * N + other * n + 5, -1
        glob[130], loc[130] = -7, -1
        rows[p, :counts[p]], local[p, :counts[p]] = glob, loc
    rows, local = rows.cuda(), local.cuda()
    d_counts = torch.tensor(counts, dtype=torch.int64, device="cuda")
    coefs = [(clips[p], 1.0 / counts[p], (0.5 + 0.25 * p) / counts[p], (0.01 * (p + 1)) / counts[p]) for p in range(P)]
    grad, ok_g = _guarded((P, pop.grad_stride), 12345.0)
    outs = [_guarded((T, N), -777.0) for _ in range(3)]
    pop.scratch = torch.full_like(pop.scratch, 0xA5)         # its contents are irrelevant
    pop.ppo_backward(feats, ctrs, acts, logp_old, adv, target, rows, d_counts, coefs, out=grad, logp=outs[0][0],
                     value=outs[1][0], entropy=outs[2][0])
    assert ok_g() and all(ok() for _, ok in outs)
    for p in range(P):
        sl = slice(p * n, (p + 1) * n)
        env_p = _env(n, base=p * n)
        tc = PolicyTrainTC(env_p, pols[p])
        c = lambda x: x[:, sl].contiguous()
        mine = [torch.full((T, n), -777.0, device="cuda") for _ in range(3)]
        want = tc.ppo_backward(c(feats), ctrs, c(acts), c(logp_old), c(adv), c(target), local[p], d_counts[p:p + 1], *coefs[p],
                               logp=mine[0], value=mine[1], entropy=mine[2])
        assert torch.equal(grad[p, :tc.n_params], want), p
        assert bool((grad[p, tc.n_params:] == 12345.0).all())   # the stride's padding is not written
        for (got, _), w in zip(outs, mine):
            assert torch.equal(got[:, sl], w), p
        env_p.close()
    env.close()


def _hps():
    return [{"lr": 3e-4, "gamma": 0.99, "lam": 0.95, "clip_eps": 0.2},
            {"lr": 1e-3, "gamma": 0.9, "lam": 0.8, "clip_eps": 0.1, "vf_coef": 1.0, "ent_coef": 0.05, "max_grad_norm": 0.1},
            {"lr": 5e-5, "gamma": 0.999, "lam": 0.97, "clip_eps": 0.3, "vf_coef": 0.25, "ent_coef": 0.0, "max_grad_norm": 2.0}]


KW = dict(horizon=T, epochs=2, minibatches=3)              # 4,096 rows per member: minibatches of 1,365 and 1,366


def _population(pols, members=P, seed=5):
    from wab_gym_b200.population import PPOPopulation
    pop = PPOPopulation(_env(members * n, seed=seed), members, _hps()[:members], policies=[copy.deepcopy(q) for q in pols], **KW)
    pop.sample_seed = 4242
    return pop


def _standalone(pol, p, seed=5):
    from wab_gym_b200.ppo import PPOTrainer
    tr = PPOTrainer(_env(n, base=p * n, seed=seed), copy.deepcopy(pol), **KW, **_hps()[p])
    tr.sample_seed = 4242
    return tr


def _same_member(pop, p, tr, stats=None, want=None):
    for a, b in zip(pop.policies[p].parameters(), tr.policy.parameters()):
        assert torch.equal(a, b)
    sa, sb = pop.optimizers[p].state_dict(), tr.optimizer.state_dict()
    assert sa["param_groups"] == sb["param_groups"]
    for k in sa["state"]:
        for key in ("step", "exp_avg", "exp_avg_sq"):
            assert torch.equal(sa["state"][k][key], sb["state"][k][key])
    sl = slice(p * n, (p + 1) * n)
    for key, v in tr.last_batch.items():
        if key in ("counters",):
            assert torch.equal(pop.last_batch[key], v)
        elif key in pop.last_batch:
            got = pop.last_batch[key][sl] if key == "bootstrap" else pop.last_batch[key][:, sl]
            assert torch.equal(got, v), key
    if stats is not None:
        for key, v in want.items():
            assert torch.equal(stats[key][p], v), key


def test_population_trains_each_member_as_its_standalone_trainer():
    env0 = _env(n)
    pols = _policies(env0, seed=7)
    env0.close()
    pop = _population(pols)
    stats = [pop.train_iteration() for _ in range(2)]
    for s in stats:
        assert all(v.shape == (P, 6) for k, v in s.items() if k != "mean_reward") and s["mean_reward"].shape == (P,)
    for p in range(P):
        tr = _standalone(pols[p], p)
        want = [tr.train_iteration() for _ in range(2)]
        for s, w in zip(stats, want):
            for key, v in w.items():
                assert torch.equal(s[key][p], v), (p, key)
        _same_member(pop, p, tr)
    # the members took different paths
    assert not torch.equal(pop.policies[0].affine1.weight, pop.policies[1].affine1.weight)


def test_a_population_of_one_is_ppo_trainer():
    env0 = _env(n)
    pols = _policies(env0, seed=9)
    env0.close()
    pop = _population(pols[:1], members=1)
    tr = _standalone(pols[0], 0)
    s, w = pop.train_iteration(), tr.train_iteration()
    for key, v in w.items():
        assert torch.equal(s[key][0], v), key
    _same_member(pop, 0, tr)


def test_resume_member_state_and_exploit():
    env0 = _env(n)
    pols = _policies(env0, seed=13)
    env0.close()
    a = _population(pols)
    a.train_iteration()
    sd = a.state_dict()
    msd = [a.member_state_dict(p) for p in range(P)]
    want = a.train_iteration()
    b = _population(_policies(_env(n), seed=99))           # other weights, other hyper-parameters' Adam state
    b.load_state_dict(sd)
    got = b.train_iteration()
    for key, v in want.items():
        assert torch.equal(got[key], v), key                  # resumed bit for bit (and two runs agree)
    for p in range(P):
        assert all(torch.equal(x, y) for x, y in zip(a.policies[p].parameters(), b.policies[p].parameters()))
    # member 1 continues as a standalone PPOTrainer
    tr = _standalone(pols[1], 1)
    tr.load_state_dict(msd[1])
    w1 = tr.train_iteration()
    for key, v in w1.items():
        assert torch.equal(want[key][1], v), key
    _same_member(a, 1, tr)
    # exploit: member 0 takes member 2's policy, Adam state and hyper-parameters; its envs stay where they were
    before = a.env.save_state(torch.arange(0, n)).records.clone()
    a.load_member_state_dict(0, a.member_state_dict(2))
    assert all(torch.equal(x, y) for x, y in zip(a.policies[0].parameters(), a.policies[2].parameters()))
    assert a.hyperparameters[0] == a.hyperparameters[2]
    s0, s2 = a.optimizers[0].state_dict(), a.optimizers[2].state_dict()
    assert s0["param_groups"][0]["lr"] == s2["param_groups"][0]["lr"]
    assert all(torch.equal(s0["state"][k]["exp_avg"], s2["state"][k]["exp_avg"]) for k in s0["state"])
    assert torch.equal(a.env.save_state(torch.arange(0, n)).records, before)
    assert a._tc._packed_versions[0] == a._tc._versions(0)  # member 0 was re-packed by the load
    a._tc.refresh([2])                                        # member 2's last Adam step is packed at its next use
    for buf in (a._tc.packed1, a._tc.packed3t, a._tc.bias2, a._tc.w_heads):
        assert torch.equal(buf[0], buf[2])


def test_an_iteration_never_synchronises():
    env0 = _env(n)
    pols = _policies(env0, seed=21)
    env0.close()
    pop = _population(pols)
    pop.train_iteration()                                    # first calls: allocations, module loads
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = pop.train_iteration()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert out["grad_norm"].shape == (P, 6)


def test_abi_refusals():
    from wab_gym_b200 import _lib
    from wab_gym_b200.policy import PolicyPopulationTC
    L = _lib.load()
    env = _env(P * n)
    env.reset()
    pop = PolicyPopulationTC(env, _policies(env))
    vp = ctypes.c_void_p
    acts = torch.empty(P * n, dtype=torch.uint8, device="cuda")
    A = env.n_actions

    def fwd(members=P, rows=n, heads=True):
        return L.wab_policy_forward_population(env._h, env.last_features.data_ptr(), members, rows, pop.packed1.data_ptr(),
                                               pop.bias1.data_ptr(), pop.packed2.data_ptr(), pop.bias2.data_ptr(), 150,
                                               pop.packed3.data_ptr(), pop.bias3.data_ptr(),
                                               pop.w_heads.data_ptr() if heads else None, pop.b_heads.data_ptr(), A, 0.01,
                                               0.01, -4.0, 4.0, 1, None, acts.data_ptr(), None, None, None, None, None)
    assert fwd() == 0
    assert fwd(members=0) == 2 and fwd(members=65) == 2
    assert fwd(rows=100) == 2 and fwd(rows=0) == 2
    assert fwd(heads=False) == 1

    f = torch.zeros(1, P * n, 28, dtype=torch.uint8, device="cuda")
    ctr = torch.ones(1, dtype=torch.int64, device="cuda")
    a1 = torch.zeros(1, P * n, dtype=torch.uint8, device="cuda")
    z = torch.zeros(1, P * n, device="cuda")
    rows = torch.zeros(P, 4, dtype=torch.int32, device="cuda")
    counts = torch.full((P,), 4, dtype=torch.int64, device="cuda")
    grad = torch.empty(P, pop.grad_stride, device="cuda")

    def bwd(members=P, n_envs=P * n, coefs=None, rows_ptr=True, list_len=4, scratch_bytes=None):
        c = coefs if coefs is not None else [0.2, 1.0, 0.5, 0.01] * max(members, P)
        arr = (ctypes.c_float * len(c))(*c)
        return L.wab_policy_ppo_backward_population(
            env._h, f.data_ptr(), 1, n_envs, members, ctr.data_ptr(), a1.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(),
            rows.data_ptr() if rows_ptr else None, list_len, counts.data_ptr(), pop.packed1.data_ptr(), pop.bias1.data_ptr(),
            pop.packed2.data_ptr(), pop.bias2.data_ptr(), 150, pop.packed3.data_ptr(), pop.bias3.data_ptr(),
            pop.packed2t.data_ptr(), pop.packed3t.data_ptr(), pop.w_heads.data_ptr(), pop.b_heads.data_ptr(), A, 0.01, 0.01,
            -4.0, 4.0, ctypes.cast(arr, vp), pop.scratch.data_ptr(),
            pop.scratch.numel() if scratch_bytes is None else scratch_bytes, grad.data_ptr(), None, None, None, None)
    assert bwd() == 0
    torch.cuda.synchronize()
    assert bwd(members=0) == 2 and bwd(members=65) == 2
    assert bwd(n_envs=P * n - 128 * P + P) == 2 and bwd(members=5) == 2      # n not a multiple of 128 / N not P n
    assert bwd(scratch_bytes=pop.scratch.numel() - 1) == 2 and b"population_scratch_bytes" in L.wab_last_error()
    assert bwd(coefs=[0.2, 1.0, 0.5, 0.01, 0.0, 1.0, 0.5, 0.01] + [0.2, 1.0, 0.5, 0.01]) == 2        # clip_eps <= 0
    assert bwd(coefs=[0.2, 1.0, 0.5, 0.01] * 2 + [0.2, float("nan"), 0.5, 0.01]) == 2                 # a non-finite weight
    assert bwd(list_len=-1) == 2
    assert bwd(rows_ptr=False) == 1
    assert L.wab_policy_backward_population_scratch_bytes(env._h, P) == P * L.wab_policy_backward_scratch_bytes(env._h)
    assert L.wab_policy_backward_population_scratch_bytes(env._h, 65) == 0
    assert pop.grad_stride % 64 == 0 and pop.n_params <= pop.grad_stride < pop.n_params + 64
    with pytest.raises(ValueError):
        PolicyPopulationTC(env, [pop.policies[0]] * 5)       # 768 envs are not 5 x a multiple of 128
    env.close()
