"""Population evaluation on the B200: the greedy population forward against the single-policy greedy forward, its return
codes, and ``PopulationEvaluator`` against P standalone ``Evaluator``s. Every comparison is bit for bit."""
import copy
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

P, n = 3, 256


def _policies(flat_dim, A, seed=1, members=P):
    """Different reference networks, scaled so both leaky branches, the clamp and close logits all occur."""
    from wab_gym_b200.policy import Policy
    out = []
    for p in range(members):
        torch.manual_seed(seed + 17 * p)
        pol = Policy(flat_dim, A).cuda()
        with torch.no_grad():
            for lin in (pol.affine1, pol.affine2, pol.affine3):
                lin.weight.mul_(3.0)
            pol.affine3.bias[:32] += 3.5
            pol.action_head.weight.mul_(4.0)
        out.append(pol)
    return out


@pytest.mark.parametrize("noise", [0.01, 0.0])
@pytest.mark.parametrize("A", [5, 3, 8])
@pytest.mark.parametrize("base", [0, 4096])
def test_forward_greedy_equals_the_single_policy_greedy_forward(noise, A, base):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import PolicyPopulationTC, PolicyTrunkTC, stacked_heads
    env = VecEnv(P * n, seed=5, env_id_base=base, features=True)
    env.reset()
    for _ in range(7):
        env.step(torch.randint(0, env.n_actions, (P * n,), device="cuda").to(torch.uint8))
    pols = _policies(env.flat_dim, A)
    pop = PolicyPopulationTC(env, pols)
    feats = env.last_features.clone()
    ctr = torch.full((1,), 9, dtype=torch.int64, device="cuda")
    N = P * n
    acts, value, probs, logp, z3 = (torch.full((N,), 250, dtype=torch.uint8, device="cuda"), torch.empty(N, device="cuda"),
                                    torch.empty(N, A, device="cuda"), torch.empty(N, device="cuda"),
                                    torch.empty(N, 128, device="cuda"))
    pop.forward_greedy(feats, acts, value=value, probs=probs, logp=logp, noise_scale=noise, counter=ctr, z3=z3)
    assert int(acts.max()) < A
    for p in range(P):
        sl = slice(p * n, (p + 1) * n)
        env_p = VecEnv(n, seed=5, env_id_base=base + p * n, features=True)
        tc = PolicyTrunkTC(env_p, pols[p])
        a, v, pr, lp, z = (torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, device="cuda"),
                           torch.empty(n, A, device="cuda"), torch.empty(n, device="cuda"), torch.empty(n, 128, device="cuda"))
        tc.forward_greedy(feats[sl].contiguous(), stacked_heads(pols[p]), a, value=v, probs=pr, logp=lp, noise_scale=noise,
                          counter=ctr, z3=z)
        assert torch.equal(acts[sl], a) and torch.equal(value[sl], v) and torch.equal(probs[sl], pr)
        assert torch.equal(logp[sl], lp) and torch.equal(z3[sl], z)
        env_p.close()
    assert not torch.equal(value[:n], value[n:2 * n])
    env.close()


def test_refusals_return_the_sampling_calls_codes():
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import PolicyPopulationTC, _ptr
    env = VecEnv(P * n, seed=5, features=True)
    env.reset()
    pop = PolicyPopulationTC(env, _policies(env.flat_dim, env.n_actions))
    L, A = env.lib, env.n_actions
    acts = torch.empty(P * n, dtype=torch.uint8, device="cuda")
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def both(members=P, rows=n, heads=pop.w_heads, actions=acts, n_actions=A, hidden=150):
        w = (env._h, _ptr(env.last_features), members, rows, _ptr(pop.packed1), _ptr(pop.bias1), _ptr(pop.packed2),
             _ptr(pop.bias2), hidden, _ptr(pop.packed3), _ptr(pop.bias3), _ptr(heads), _ptr(pop.b_heads), n_actions, 0.01, 0.01,
             -4.0, 4.0)
        tail = (None, _ptr(actions), None, None, None, None, s)
        return L.wab_policy_act_population(*w, *tail), L.wab_policy_forward_population(*w, 3, *tail)

    assert both() == (0, 0)
    for kw, code in ((dict(members=0), 2), (dict(members=65), 2), (dict(rows=100), 2), (dict(rows=0), 2),
                     (dict(heads=None), 1), (dict(actions=None), 1), (dict(n_actions=9), 2), (dict(n_actions=0), 2),
                     (dict(hidden=128), 3)):
        act, fwd = both(**kw)
        assert act == fwd == code, kw
    with pytest.raises(ValueError, match="features"):
        pop.forward_greedy(env.last_features[:n], acts)
    with pytest.raises(ValueError, match="actions"):
        pop.forward_greedy(env.last_features, acts[:n])
    with pytest.raises(ValueError, match="probs"):
        pop.forward_greedy(env.last_features, acts, probs=torch.empty(P * n, A + 1, device="cuda"))
    env.close()


def _state(pols):
    return [{k: v.detach().clone() for k, v in p.state_dict().items()} for p in pols]


@pytest.mark.parametrize("greedy", [True, False])
def test_population_evaluator_equals_standalone_evaluators(greedy):
    from wab_gym_b200 import Evaluator, PopulationEvaluator
    k, base = 2, 640
    pe = PopulationEvaluator(P, n, seed=3, env_id_base=base, episodes_per_env=k)
    pols = _policies(pe.flat_dim, pe.n_actions, seed=4)
    before = _state(pols)
    got = pe.evaluate(pols, greedy=greedy)
    assert len(got) == P
    ev = Evaluator(n, seed=3, env_id_base=base, episodes_per_env=k)
    for p in range(P):
        want = ev.evaluate(pols[p], greedy=greedy)
        for g, w in zip(got[p], want):
            assert g.dtype == w.dtype and torch.equal(g, w), p
    assert not torch.equal(got[0].returns, got[1].returns)
    # the policies are only read; a second call repeats the first
    for b, a in zip(before, _state(pols)):
        assert all(torch.equal(b[key], a[key]) for key in b)
    assert all(prm.grad is None for pol in pols for prm in pol.parameters())
    again = pe.evaluate(pols, greedy=greedy)
    for g, a in zip(got, again):
        assert all(torch.equal(x, y) for x, y in zip(g, a))
    pe.close()
    ev.close()


def test_equal_policies_give_equal_results_and_noise_off_runs():
    from wab_gym_b200 import PopulationEvaluator
    pe = PopulationEvaluator(2, 128, seed=9)
    pol = _policies(pe.flat_dim, pe.n_actions, members=1)[0]
    for noise in (True, False):
        a, b = pe.evaluate([pol, copy.deepcopy(pol)], noise=noise)
        assert all(torch.equal(x, y) for x, y in zip(a, b))
    pe.close()


def test_refusals():
    from wab_gym_b200 import PopulationEvaluator
    for kw, match in ((dict(members=0), "1 to 64"), (dict(members=65), "1 to 64"), (dict(envs_per_member=100), "128"),
                      (dict(group=object()), "group")):
        args = dict(members=2, envs_per_member=128)
        args.update(kw)
        with pytest.raises(ValueError, match=match):
            PopulationEvaluator(**args)
    pe = PopulationEvaluator(2, 128)
    pols = _policies(pe.flat_dim, pe.n_actions, members=3)
    with pytest.raises(ValueError, match="one policy per member"):
        pe.evaluate(pols)
    with pytest.raises(ValueError, match="same action count"):
        pe.evaluate([pols[0], _policies(pe.flat_dim, 4, members=1)[0]])
    pe.close()


def test_the_step_loop_never_synchronises():
    from wab_gym_b200 import PopulationEvaluator
    pe = PopulationEvaluator(4, 128, seed=2)
    pols = _policies(pe.flat_dim, pe.n_actions, members=4)
    for greedy in (True, False):
        pe.restore(pols)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            pe.play(greedy=greedy)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        torch.cuda.synchronize()
    pe.close()
