"""Evaluation on the GPU: the greedy tail of the one-launch forward (``wab_policy_act`` / ``forward_greedy``) against
``torch.argmax`` of the evaluated logits and against the sampler's arithmetic, and ``Evaluator`` against a hand-written
loop, replayed with common random numbers, isolated from a trainer, without host synchronisation and over two ranks."""
import ctypes
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

from tests.test_evaluate import _loop

pytestmark = pytest.mark.gpu


def _setup(n, env_id_base=0, seed=1, options=None, warm=5):
    """A handle with env_id_base, features after a few random steps, a policy whose actions spread, its packed copy."""
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy, PolicyTrainTC
    env = VecEnv(n, game_options=options, seed=seed, features=True, env_id_base=env_id_base)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(warm):
        env.step(torch.randint(0, env.n_actions, (n,), device="cuda", generator=g).to(torch.uint8))
    torch.manual_seed(seed)
    pol = Policy(env.flat_dim, env.n_actions).cuda()
    with torch.no_grad():
        for lin in (pol.affine1, pol.affine2, pol.affine3):
            lin.weight.mul_(3.0)
        pol.action_head.weight.mul_(4.0)
    return env, pol, PolicyTrainTC(env, pol)


def _outputs(n, A):
    return (torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, device="cuda"),
            torch.empty(n, A, device="cuda"), torch.empty(n, device="cuda"))


@pytest.mark.parametrize("noise", [0.01, 0.0])
def test_greedy_is_the_argmax_of_the_logits(noise):
    n = 1003                                                            # ragged: not a multiple of 128
    env, pol, tc = _setup(n, env_id_base=777)
    feats = env.last_features.clone()
    ctr = torch.full((1,), 41, dtype=torch.int64, device="cuda")
    acts, v, p, lp = _outputs(n, env.n_actions)
    tc.forward_greedy(feats, tc.heads, acts, value=v, probs=p, logp=lp, noise_scale=noise, counter=ctr)
    with torch.no_grad():
        logits, value = tc.logits_and_value(feats[None].contiguous(), ctr.clone(), noise_scale=noise)
    assert torch.equal(acts.long(), torch.argmax(logits, -1))
    assert torch.equal(v, value)
    assert len(torch.unique(acts)) > 1                                  # the argmax is not a constant here
    env.close()


def test_exact_ties_go_to_the_lowest_index():
    n = 1003
    env, pol, tc = _setup(n, env_id_base=5)
    with torch.no_grad():                                               # rows 1 and 3 identical and dominant: bit-equal logits
        pol.action_head.weight[3].copy_(pol.action_head.weight[1])
        pol.action_head.bias[1] = 500.0
        pol.action_head.bias[3] = 500.0
    tc.refresh()
    ctr = torch.full((1,), 7, dtype=torch.int64, device="cuda")
    acts, v, p, lp = _outputs(n, env.n_actions)
    tc.forward_greedy(env.last_features, tc.heads, acts, probs=p, noise_scale=0.01, counter=ctr)
    with torch.no_grad():
        logits, _ = tc.logits_and_value(env.last_features[None].contiguous(), ctr.clone(), noise_scale=0.01)
    tied = logits[:, 1] == logits[:, 3]
    top = logits.max(-1).values
    assert bool(tied.all()) and bool((logits[:, 1] == top).all())
    assert bool((acts == 1).all()) and torch.equal(acts.long(), torch.argmax(logits, -1))
    assert torch.equal(p[:, 1], p[:, 3])
    env.close()


@pytest.mark.parametrize("noise", [0.01, 0.0])
def test_same_arithmetic_as_the_sampler(noise):
    n = 1500
    env, pol, tc = _setup(n, env_id_base=300)
    feats = env.last_features.clone()
    ctr = torch.full((1,), 99, dtype=torch.int64, device="cuda")
    A = env.n_actions
    ga, gv, gp, glp = _outputs(n, A)
    gz = torch.empty(n, 128, device="cuda")
    tc.forward_greedy(feats, tc.heads, ga, value=gv, probs=gp, logp=glp, noise_scale=noise, counter=ctr, z3=gz)
    sa, sv, sp, slp = _outputs(n, A)
    sz = torch.empty(n, 128, device="cuda")
    tc.forward_sample(feats, tc.heads, sa, value=sv, probs=sp, logp=slp, noise_scale=noise, counter=ctr, seed=17, z3=sz)
    assert torch.equal(gv, sv) and torch.equal(gp, sp) and torch.equal(gz, sz)
    same = sa == ga
    assert 0 < int(same.sum()) < n                                      # both kinds of row occur
    assert torch.equal(glp[same], slp[same])
    with torch.no_grad():
        logits, _ = tc.logits_and_value(feats[None].contiguous(), ctr.clone(), noise_scale=noise)
    want = torch.log_softmax(logits, -1).gather(1, ga.long()[:, None]).squeeze(1)
    assert float((glp - want).abs().max()) <= 1e-6
    # the sampling seed moves the samples and nothing of the greedy output
    other = torch.empty_like(sa)
    tc.forward_sample(feats, tc.heads, other, noise_scale=noise, counter=ctr, seed=18)
    assert not torch.equal(other, sa)
    again = _outputs(n, A)
    tc.forward_greedy(feats, tc.heads, again[0], value=again[1], probs=again[2], logp=again[3], noise_scale=noise, counter=ctr)
    for x, y in zip(again, (ga, gv, gp, glp)):
        assert torch.equal(x, y)
    env.close()


def _abi(fn, tc, env, features, rows, bufs, **kw):
    """wab_policy_act or wab_policy_forward (fn) through the C ABI with every argument overridable."""
    from wab_gym_b200.vec_env import _ptr
    w, b = tc.heads
    a = dict(h=env._h, feats=_ptr(features), n=rows, p1=_ptr(tc.packed), b1=_ptr(tc.bias), p2=_ptr(tc.packed2), b2=_ptr(tc.bias2),
             hidden2=150, p3=_ptr(tc.packed3), b3=_ptr(tc.bias3), wh=_ptr(w), bh=_ptr(b), A=w.shape[0] - 1, ctr=_ptr(bufs["ctr"]),
             actions=bufs["actions"], value=bufs["value"], probs=bufs["probs"], logp=bufs["logp"], z3=bufs["z3"])
    a.update(kw)
    head = (a["h"], a["feats"], a["n"], a["p1"], a["b1"], a["p2"], a["b2"], a["hidden2"], a["p3"], a["b3"], a["wh"], a["bh"],
            a["A"], 0.01, 0.01, -4.0, 4.0)
    tail = (a["ctr"], a["actions"], a["value"], a["probs"], a["logp"], a["z3"], None)
    if fn == "act":
        return tc.lib.wab_policy_act(*head, *tail)
    return tc.lib.wab_policy_forward(*head, 23, *tail)


def test_deterministic_in_bounds_and_refuses_what_the_sampler_refuses():
    n, guard = 1003, 4096
    env, pol, tc = _setup(n, env_id_base=64)
    A = env.n_actions
    feats = env.last_features.clone()
    ctr = torch.full((1,), 3, dtype=torch.int64, device="cuda")
    fills = {"actions": 0xAB, "value": -777.0, "probs": -777.0, "logp": -777.0, "z3": -777.0}
    sizes = {"actions": n, "value": n, "probs": n * A, "logp": n, "z3": n * 128}
    runs = []
    for _ in range(2):
        bufs = {k: torch.full((sizes[k] + 2 * guard,), fills[k], dtype=torch.uint8 if k == "actions" else torch.float32,
                              device="cuda") for k in sizes}
        ptrs = {k: ctypes.c_void_p(bufs[k][guard:].data_ptr()) for k in bufs}
        assert _abi("act", tc, env, feats, n, {**ptrs, "ctr": ctr}) == 0
        torch.cuda.synchronize()
        for k, buf in bufs.items():
            assert bool((buf[:guard] == fills[k]).all()) and bool((buf[guard + sizes[k]:] == fills[k]).all()), k
            assert not bool((buf[guard:guard + sizes[k]] == fills[k]).all()), k
        runs.append({k: buf[guard:guard + sizes[k]].clone() for k, buf in bufs.items()})
    for k in sizes:
        assert torch.equal(runs[0][k], runs[1][k]), k                  # two launches are bit-identical
    # refusals: the same return code as wab_policy_forward for every bad argument (1 NULL, 2 CONFIG, 3 UNSUPPORTED)
    out = {"actions": torch.empty(n, dtype=torch.uint8, device="cuda"), "value": torch.empty(n, device="cuda"),
           "probs": torch.empty(n, A, device="cuda"), "logp": torch.empty(n, device="cuda"),
           "z3": torch.empty(n, 128, device="cuda")}
    ptrs = {k: ctypes.c_void_p(v.data_ptr()) for k, v in out.items()}
    ptrs["ctr"] = ctr
    off = lambda t, b: ctypes.c_void_p(t.data_ptr() + b)
    cases = [({}, 0), ({"value": None, "probs": None, "logp": None, "z3": None}, 0), ({"n": 0}, 0)]
    cases += [({k: None}, 1) for k in ("h", "feats", "p1", "b1", "p2", "b2", "p3", "b3", "wh", "bh", "actions")]
    cases += [({"A": 0}, 2), ({"A": 9}, 2), ({"hidden2": 140}, 3), ({"z3": off(out["z3"], 4)}, 2),
              ({"feats": off(feats, 1)}, 2), ({"p1": off(tc.packed, 8)}, 2), ({"p2": off(tc.packed2, 4)}, 2),
              ({"p3": off(tc.packed3, 8)}, 2)]
    for kw, want in cases:
        got_act = _abi("act", tc, env, feats, n, ptrs, **kw)
        got_fwd = _abi("forward", tc, env, feats, n, ptrs, **kw)
        assert got_act == got_fwd == want, (kw, got_act, got_fwd)
    torch.cuda.synchronize()
    env.close()


# ---- Evaluator --------------------------------------------------------------------------------------------------------

def _policy(env, seed, scale=3.0):
    from wab_gym_b200.policy import Policy
    torch.manual_seed(seed)
    pol = Policy(env.flat_dim, env.n_actions)
    with torch.no_grad():
        for lin in (pol.affine1, pol.affine2, pol.affine3):
            lin.weight.mul_(scale)
        pol.action_head.weight.mul_(4.0)
    return pol


def _hand_loop(n, seed, pol, greedy, noise, steps, sample_seed, env_id_base=0):
    """What Evaluator.evaluate promises, written out: a fresh env of the same seed, the policy's greedy or sampled
    action from a counter starting at 0, env.step; reward, done and info read back on the host."""
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import PolicyTrunkTC, stacked_heads
    env = VecEnv(n, seed=seed, features=True, emit_grids=False, env_id_base=env_id_base)
    env.reset()
    p = pol.cuda() if next(pol.parameters()).device.type != "cuda" else pol
    tc, heads = PolicyTrunkTC(env, p), stacked_heads(p)
    ctr = torch.zeros(1, dtype=torch.int64, device="cuda")
    acts = torch.empty(n, dtype=torch.uint8, device="cuda")
    rec = {"reward": [], "done": [], "info": [], "features": [env.last_features.cpu()]}
    for _ in range(steps):
        ctr += 1
        if greedy:
            tc.forward_greedy(env.last_features, heads, acts, noise_scale=0.01 if noise else 0.0, counter=ctr)
        else:
            tc.forward_sample(env.last_features, heads, acts, noise_scale=0.01 if noise else 0.0, counter=ctr, seed=sample_seed)
        _, r, d, info = env.step(acts)
        rec["reward"].append(r.cpu()); rec["done"].append(d.cpu()); rec["info"].append(info["info"].cpu())
        rec["features"].append(env.last_features.cpu())
    env.close()
    return {k: torch.stack(v) for k, v in rec.items()}


@pytest.mark.parametrize("greedy", [True, False])
def test_evaluator_equals_a_hand_loop(greedy):
    from wab_gym_b200 import Evaluator
    n, seed, k = 700, 3, 2
    ev = Evaluator(n, seed=seed, episodes_per_env=2)
    pol = _policy(ev.env, 4)
    res = ev.evaluate(pol, greedy=greedy)
    rec = _hand_loop(n, seed, pol, greedy, True, ev.steps, ev.sample_seed)
    want = _loop(rec["reward"], rec["done"], rec["info"], k)
    assert res.returns.shape == (n, k) and res.first_features.shape == (n, k, 28)
    assert res.returns.tolist() == want["returns"] and res.lengths.tolist() == want["lengths"]
    assert res.outcome.tolist() == want["outcome"] and res.eats.tolist() == want["eats"]
    # the first observation of each episode: the start, then the observation after each done
    d = rec["done"]
    for nn_ in range(0, n, 37):
        ends = torch.nonzero(d[:, nn_]).squeeze(1).tolist()
        starts = [0] + [t + 1 for t in ends[:k - 1]]
        for j, t in enumerate(starts):
            assert torch.equal(res.first_features[nn_, j], rec["features"][t, nn_]), (nn_, j)
    s = res.summary()
    assert s["episodes"] == n * k and abs(s["finished"] + s["starved"] + s["killed"] - 1.0) < 1e-12
    ev.close()


def test_replayable_with_common_random_numbers():
    from wab_gym_b200 import Evaluator
    ev = Evaluator(900, seed=5, episodes_per_env=2)
    a, b = _policy(ev.env, 1).cuda(), _policy(ev.env, 2, scale=1.0).cuda()
    ra, rb, ra2 = ev.evaluate(a), ev.evaluate(b), ev.evaluate(a)
    for x, y in zip(ra, ra2):
        assert torch.equal(x, y)
    assert not torch.equal(ra.returns, rb.returns)                      # the policies play differently ...
    assert torch.equal(ra.first_features, rb.first_features)            # ... from the same episode starts
    for greedy, noise in ((False, True), (True, False)):
        r1, r2 = ev.evaluate(a, greedy=greedy, noise=noise), ev.evaluate(a, greedy=greedy, noise=noise)
        for x, y in zip(r1, r2):
            assert torch.equal(x, y)
        assert torch.equal(r1.first_features, ra.first_features)
    ev.close()


def test_evaluating_between_iterations_leaves_training_bit_identical():
    from wab_gym_b200 import Evaluator, VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    from wab_gym_b200.sharding import _bit_equal

    def trainer():
        env = VecEnv(512, seed=9, features=True, emit_grids=False)
        torch.manual_seed(0)
        return PPOTrainer(env, Policy(env.flat_dim, env.n_actions), horizon=16, epochs=2, minibatches=2)

    plain, watched = trainer(), trainer()
    ev = Evaluator(300, seed=9)
    for _ in range(3):
        plain.train_iteration()
        watched.train_iteration()
        ev.evaluate(watched.policy)
        ev.evaluate(watched.policy, greedy=False)
    for p, q in zip(plain.policy.parameters(), watched.policy.parameters()):
        assert torch.equal(p, q)
    assert _bit_equal(plain.optimizer.state_dict(), watched.optimizer.state_dict())
    assert _bit_equal(plain.state_dict(), watched.state_dict())
    plain.train_iteration()
    watched.train_iteration()
    assert all(torch.equal(p, q) for p, q in zip(plain.policy.parameters(), watched.policy.parameters()))
    for tr in (plain, watched):
        tr.env.close()
    ev.close()


def test_the_step_loop_never_synchronises():
    from wab_gym_b200 import Evaluator
    ev = Evaluator(640, seed=2)
    pol = _policy(ev.env, 3).cuda()
    for greedy in (True, False):
        ev.restore(pol)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            ev.play(greedy=greedy)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        torch.cuda.synchronize()
    ev.close()


# ---- two ranks --------------------------------------------------------------------------------------------------------

N_TOTAL, SEED, K = 1001, 13, 2                 # ragged shards: 501 + 500


def _eval_all(ev, pol):
    return [ev.evaluate(pol, greedy=g, noise=z) for g, z in ((True, True), (False, True), (True, False))]


def _worker(rank, world, port, backend, outdir):
    import torch.distributed as dist
    from wab_gym_b200 import Evaluator
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=world)
    ev = Evaluator(N_TOTAL, seed=SEED, episodes_per_env=K, group=dist.group.WORLD,
                   device=torch.device("cuda", torch.cuda.current_device()))
    assert ev.env.num_envs == (501 if rank == 0 else 500) and ev.env.env_id_base == (0 if rank == 0 else 501)
    out = _eval_all(ev, _policy(ev.env, 6))                             # a CPU policy: evaluate copies it over
    torch.save([tuple(r) for r in out], os.path.join(outdir, "eval%d.pt" % rank))
    ev.close()
    dist.barrier()
    dist.destroy_process_group()


def _check_two_ranks(backend, tmp_path):
    from wab_gym_b200 import Evaluator
    ev = Evaluator(N_TOTAL, seed=SEED, episodes_per_env=K)
    want = _eval_all(ev, _policy(ev.env, 6))
    ev.close()
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, backend, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        got = torch.load(os.path.join(str(tmp_path), "eval%d.pt" % r))
        for g, w in zip(got, want):
            for x, y in zip(g, w):
                assert torch.equal(x, y), r


def test_two_ranks_on_one_gpu_over_gloo(tmp_path):
    _check_two_ranks("gloo", tmp_path)


def test_two_ranks_on_two_gpus_over_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL needs two visible GPUs; this machine shows %d" % torch.cuda.device_count())
    _check_two_ranks("nccl", tmp_path)
