"""Data-parallel populations on the B200: blocked handles (every block equals a standalone ``VecEnv`` at its ids, byte for
byte), the population kernels on a blocked handle, the population gradient in fp64, and ``PPOPopulation`` /
``PopulationEvaluator`` / ``PopulationBasedTraining`` over two ranks (gloo on one GPU, NCCL on two when visible)."""
import copy
import ctypes
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

K, C, STRIDE, BASE, STEPS = 3, 200, 1000, 37, 300


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _outputs(env, obs, reward, done, info):
    out = [obs.food, obs.role, obs.status, reward, done, info["info"]]
    if obs.grids is not None:
        out.append(obs.grids)
    if env.with_features:
        out.append(env.last_features)
    return out


@pytest.mark.parametrize("kind", ["default", "lookout_off", "generic"])
def test_each_block_equals_a_standalone_env(kind):
    from wab_gym_b200 import VecEnv
    opts = {"width": 13, "height": 13} if kind == "generic" else {"lookout_only": False} if kind == "lookout_off" else None
    kw = dict(features=kind != "generic")
    blk = VecEnv(K * C, game_options=opts, seed=7, env_id_base=BASE, blocks=K, block_stride=STRIDE, **kw)
    alone = [VecEnv(C, game_options=opts, seed=7, env_id_base=BASE + k * STRIDE, **kw) for k in range(K)]
    assert blk.generic_kernels == (kind == "generic")
    blk.reset()
    for a in alone:
        a.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(STEPS):
        acts = torch.randint(0, blk.n_actions, (K * C,), generator=gen, device="cuda", dtype=torch.int64).to(torch.uint8)
        got = _outputs(blk, *blk.step(acts))
        for k, a in enumerate(alone):
            want = _outputs(a, *a.step(acts[k * C:(k + 1) * C]))
            for g, w in zip(got, want):
                assert torch.equal(g[k * C:(k + 1) * C], w), (kind, t, k)
    st = blk.save_state()
    assert st.env_ids.tolist() == [BASE + k * STRIDE + j for k in range(K) for j in range(C)]
    for k, a in enumerate(alone):
        sa = a.save_state()
        assert torch.equal(st.records[k * C:(k + 1) * C], sa.records) and torch.equal(st.env_ids[k * C:(k + 1) * C], sa.env_ids)
    assert blk.stats()["killed"] > 0
    for env in [blk] + alone:
        env.close()


def test_state_dict_round_trips_and_maps_ids_to_slots():
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.vec_env import EnvStates
    mk = lambda: VecEnv(K * C, seed=7, env_id_base=BASE, blocks=K, block_stride=STRIDE, features=True)
    a = mk()
    a.reset()
    gen = torch.Generator(device="cuda").manual_seed(5)
    step = lambda: torch.randint(0, a.n_actions, (K * C,), generator=gen, device="cuda", dtype=torch.int64).to(torch.uint8)
    for _ in range(40):
        a.step(step())
    sd = a.state_dict()
    assert sd["env_ids"].tolist() == a.global_ids().tolist()
    b = mk()
    b.load_state_dict(sd)
    one = VecEnv(C, seed=7, env_id_base=BASE + STRIDE, features=True)        # block 1 alone, from the same dict
    one.load_state_dict(sd)
    c = mk()                                                                  # load_state without slots: ids -> slots
    shuffled = torch.randperm(K * C, generator=torch.Generator().manual_seed(1))
    st = a.save_state()
    c.load_state(EnvStates(st.records[shuffled.cuda()], st.env_ids[shuffled], st.fingerprint))
    for _ in range(30):
        acts = step()
        ra, rb, rc = (_outputs(e, *e.step(acts)) for e in (a, b, c))
        r1 = _outputs(one, *one.step(acts[C:2 * C]))
        for x, y, z, w in zip(ra, rb, rc, r1):
            assert torch.equal(x, y) and torch.equal(x, z) and torch.equal(x[C:2 * C], w)
    with pytest.raises(ValueError, match="outside"):                          # an id in the gap between blocks
        a.load_state(EnvStates(st.records[:1], torch.tensor([BASE + C]), st.fingerprint))
    for e in (a, b, c, one):
        e.close()


def test_set_blocks_refusals_and_return_codes():
    from wab_gym_b200 import VecEnv
    env = VecEnv(4 * 128, seed=1, features=True)
    lib, h = env.lib, env._h
    assert lib.wab_vec_set_blocks(h, 3, 0) == 2                  # does not divide n_envs
    assert lib.wab_vec_set_blocks(h, 0, 0) == 2
    assert lib.wab_vec_set_blocks(h, 4, 127) == 2                # 0 < stride < N / blocks: overlapping ids
    assert lib.wab_vec_set_blocks(h, 4, -1) == 2
    assert lib.wab_vec_set_blocks(None, 4, 128) == 1
    assert lib.wab_vec_set_blocks(h, 4, 128) == 0                # stride = block size: the plain ids
    assert lib.wab_vec_set_blocks(h, 4, 0) == 0                  # stride 0: replicas
    assert lib.wab_vec_set_blocks(h, 1, 5) == 2                  # one block of 512 ids: stride 5 would overlap
    assert lib.wab_vec_set_blocks(h, 1, 0) == 0                  # one block: the plain handle
    assert lib.wab_vec_set_blocks(h, 4, 2 ** 32) == 2            # ids 2^32 or more past env_id_base
    assert lib.wab_vec_set_blocks(h, 4, (2 ** 32 - 128) // 3 + 1) == 2
    assert lib.wab_vec_set_blocks(h, 4, (2 ** 32 - 128) // 3) == 0   # the last block ends within 2^32
    env.reset()
    assert lib.wab_vec_set_blocks(h, 4, 128) == 2                # after the first reset
    env.close()
    for kw, match in ((dict(blocks=3), "divide"), (dict(blocks=2, block_stride=100), "block_stride"),
                      (dict(blocks=2, block_stride=512, replicas=2), "not both")):
        with pytest.raises(ValueError, match=match):
            VecEnv(512, **kw)


def _policies(flat_dim, A, P, seed=1):
    from wab_gym_b200.policy import Policy
    out = []
    for p in range(P):
        torch.manual_seed(seed + 17 * p)
        pol = Policy(flat_dim, A).cuda()
        with torch.no_grad():
            for lin in (pol.affine1, pol.affine2, pol.affine3):
                lin.weight.mul_(3.0)
            pol.action_head.weight.mul_(4.0)
        out.append(pol)
    return out


def test_population_kernels_on_a_blocked_handle_and_the_fp64_gradient():
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.population import member_rows
    from wab_gym_b200.policy import PolicyPopulationTC, PolicyTrainTC
    P, c, n, f, T = 3, 256, 1024, 384, 6                            # rank holding [384, 640) of members of 1,024 envs
    env = VecEnv(P * c, seed=5, env_id_base=f, blocks=P, block_stride=n, features=True)
    env.reset()
    pols = _policies(env.flat_dim, env.n_actions, P)
    pop = PolicyPopulationTC(env, pols)
    N, A = P * c, env.n_actions
    feats = torch.empty(T, N, 28, dtype=torch.uint8, device="cuda")
    ctrs = torch.arange(50, 50 + T, dtype=torch.int64, device="cuda")
    acts = torch.empty(T, N, dtype=torch.uint8, device="cuda")
    val, lp = torch.empty(T, N, device="cuda"), torch.empty(T, N, device="cuda")
    for t in range(T):
        feats[t].copy_(env.last_features)
        pop.forward_sample(feats[t], acts[t], value=val[t], logp=lp[t], counter=ctrs[t:t + 1], seed=17)
        env.step(acts[t])
    g = torch.Generator(device="cuda").manual_seed(11)
    adv, target = torch.randn(T, N, device="cuda", generator=g), torch.randn(T, N, device="cuda", generator=g)
    logp_old = (lp + 0.3 * torch.randn(T, N, device="cuda", generator=g)).contiguous()
    perm = torch.randperm(T * c, generator=torch.Generator().manual_seed(2)).to(torch.int32).cuda()
    rows = member_rows(perm, P, c)
    counts = torch.full((P,), T * c, dtype=torch.int64, device="cuda")
    coefs = [(0.2, 1.0 / (T * c), 0.5 / (T * c), 0.01 * (p + 1) / (T * c)) for p in range(P)]
    grad = torch.full((P, pop.grad_stride), 12345.0, device="cuda")
    outs = [torch.empty(T, N, device="cuda") for _ in range(3)]
    pop.ppo_backward(feats, ctrs, acts, logp_old, adv, target, rows, counts, coefs, out=grad, logp=outs[0], value=outs[1],
                     entropy=outs[2])
    for p in range(P):                                              # member p = the single-policy calls at its ids
        sl = slice(p * c, (p + 1) * c)
        env_p = VecEnv(c, seed=5, env_id_base=p * n + f, features=True)
        tc = PolicyTrainTC(env_p, pols[p])
        cc = lambda x: x[:, sl].contiguous()
        for t in range(T):
            a, v, l = torch.empty(c, dtype=torch.uint8, device="cuda"), torch.empty(c, device="cuda"), torch.empty(c, device="cuda")
            tc.forward_sample(feats[t, sl].contiguous(), tc.heads, a, value=v, logp=l, counter=ctrs[t:t + 1], seed=17)
            assert torch.equal(a, acts[t, sl]) and torch.equal(v, val[t, sl]) and torch.equal(l, lp[t, sl]), (p, t)
        mine = [torch.empty(T, c, device="cuda") for _ in range(3)]
        want = tc.ppo_backward(cc(feats), ctrs, cc(acts), cc(logp_old), cc(adv), cc(target), perm, counts[p:p + 1], *coefs[p],
                               logp=mine[0], value=mine[1], entropy=mine[2])
        assert torch.equal(grad[p, :tc.n_params], want), p
        for got, w in zip(outs, mine):
            assert torch.equal(got[:, sl], w), p
        env_p.close()
    # the fp64 gradient: one rank's sum is the f32 gradient bit for bit; padding 0; guards untouched
    GUARD = 4096
    buf = torch.full((P * pop.grad_stride + 2 * GUARD,), -777.0, dtype=torch.float64, device="cuda")
    g64 = buf[GUARD:GUARD + P * pop.grad_stride].view(P, pop.grad_stride)
    pop.grad_f64(g64)
    assert bool((buf[:GUARD] == -777.0).all()) and bool((buf[-GUARD:] == -777.0).all())
    npar = pop.n_params
    assert bool((g64[:, npar:] == 0).all())
    summed = pop.grad_sum_ranks(g64[None].contiguous())
    assert torch.equal(summed[:, :npar], grad[:, :npar]) and bool((summed[:, npar:] == 0).all())
    assert torch.equal(g64[:, :npar].float(), grad[:, :npar])
    # refusals and return codes
    lib, h = env.lib, env._h
    f64 = lib.wab_policy_backward_population_grad_f64
    sb = pop.scratch.numel()
    assert f64(None, _ptr(pop.scratch), sb, P, A, _ptr(g64), _stream()) == 1
    assert f64(h, None, sb, P, A, _ptr(g64), _stream()) == 1
    assert f64(h, _ptr(pop.scratch), sb, P, A, None, _stream()) == 1
    assert f64(h, _ptr(pop.scratch), sb, 0, A, _ptr(g64), _stream()) == 2
    assert f64(h, _ptr(pop.scratch), sb, 65, A, _ptr(g64), _stream()) == 2
    assert f64(h, _ptr(pop.scratch), sb, P, 9, _ptr(g64), _stream()) == 3
    assert f64(h, _ptr(pop.scratch), sb - 1, P, A, _ptr(g64), _stream()) == 2
    assert f64(h, _ptr(pop.scratch), sb, P + 1, A, _ptr(g64), _stream()) == 2          # scratch of P members only
    assert f64(h, ctypes.c_void_p(pop.scratch.data_ptr() + 8), sb - 16, P, A, _ptr(g64), _stream()) == 2
    assert f64(h, _ptr(pop.scratch), sb, P, A, ctypes.c_void_p(g64.data_ptr() + 4), _stream()) == 2
    torch.cuda.synchronize()
    assert bool((buf[:GUARD] == -777.0).all()) and bool((buf[-GUARD:] == -777.0).all())
    env.close()


# ---- two ranks -------------------------------------------------------------------------------------------------------

PD, ND, TD = 2, 512, 8                                   # 2 members of 512 envs: 256 per member on each of two ranks
HPS = [{"lr": 3e-4, "clip_eps": 0.2}, {"lr": 1e-3, "gamma": 0.9, "lam": 0.8, "clip_eps": 0.1, "ent_coef": 0.05,
                                        "max_grad_norm": 0.1}]
KWD = dict(horizon=TD, epochs=2, minibatches=3)
REC = ("features", "counters", "actions", "logp", "value", "reward", "done")


def _pols():
    from wab_gym_b200 import VecEnv
    e = VecEnv(128, features=True)
    out = _policies(e.flat_dim, e.n_actions, PD, seed=21)
    e.close()
    return out


def _dp_population(pols, first, c, group, members=PD, base=0, hps=None):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.population import PPOPopulation
    env = VecEnv(members * c, seed=5, env_id_base=base + first, features=True,
                 **({"blocks": members, "block_stride": ND} if members > 1 else {}))
    pop = PPOPopulation(env, members, hps or HPS[:members], policies=[copy.deepcopy(p) for p in pols], group=group, **KWD)
    pop.sample_seed = 4242
    return pop


def _params(pop):
    return [torch.cat([prm.detach().reshape(-1) for prm in pol.parameters()]).cpu() for pol in pop.policies]


def _adam(pop):
    return [[torch.cat([st[k].reshape(-1).cpu() for st in opt.state_dict()["state"].values()]) for k in ("exp_avg", "exp_avg_sq")]
            for opt in pop.optimizers]


def _stats_cpu(s):
    return {k: v.cpu() for k, v in s.items()}


def _worker(rank, world, port, backend, outdir):
    import torch.distributed as dist
    from wab_gym_b200 import PopulationBasedTraining, PopulationEvaluator
    from wab_gym_b200.ppo import PPOTrainer
    from wab_gym_b200.sharding import merge_population_state_dicts, population_shards
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=world)
    G = dist.group.WORLD
    first, c = population_shards(ND, world)[rank]
    pols = _pols()
    out = {"first_c": (first, c)}
    # the population: first batch, two iterations, per-rank and merged checkpoints, a third iteration
    pop = _dp_population(pols, first, c, G)
    stats = [_stats_cpu(pop.train_iteration())]
    out["first"] = {k: pop.last_batch[k].cpu().clone() for k in REC}
    stats.append(_stats_cpu(pop.train_iteration()))
    out["stats"], out["params2"], out["adam2"] = stats, _params(pop), _adam(pop)
    sd = pop.state_dict()
    sds = [None] * world
    dist.all_gather_object(sds, sd, group=G)
    if rank == 0:
        torch.save(merge_population_state_dicts(sds), os.path.join(outdir, "merged2.pt"))
    pop.train_iteration()
    out["third"] = {k: pop.last_batch[k].cpu().clone() for k in REC}
    out["params3"] = _params(pop)
    pop.env.close()
    # resumed from this rank's own state dict on the same layout: the third iteration again
    res = _dp_population(pols, first, c, G)
    res.load_state_dict(sd)
    res.train_iteration()
    out["params3_resumed"] = _params(res)
    res.env.close()
    # member p = a 1-member data-parallel population on ids from p n
    for p in range(PD):
        one = _dp_population([pols[p]], first, c, G, members=1, base=p * ND, hps=[HPS[p]])
        s1 = [_stats_cpu(one.train_iteration()) for _ in range(2)]
        out["member%d" % p] = {"stats": s1, "params": _params(one), "adam": _adam(one),
                               "batch": {k: one.last_batch[k].cpu().clone() for k in one.last_batch}}
        one.env.close()
    pop2 = _dp_population(pols, first, c, G)
    for _ in range(2):
        pop2.train_iteration()
    out["pop_batch2"] = {k: pop2.last_batch[k].cpu().clone() for k in pop2.last_batch}
    pop2.env.close()
    # a 1-member population at id 0 = PPOTrainer(group)
    one = _dp_population([pols[0]], first, c, G, members=1, hps=[HPS[0]])
    from wab_gym_b200 import VecEnv
    tr = PPOTrainer(VecEnv(c, seed=5, env_id_base=first, features=True), copy.deepcopy(pols[0]), group=G, **KWD, **HPS[0])
    tr.sample_seed = 4242
    a = [_stats_cpu(one.train_iteration()) for _ in range(2)]
    b = [_stats_cpu(tr.train_iteration()) for _ in range(2)]
    out["vs_trainer"] = (a, b, _params(one)[0], torch.cat([prm.detach().reshape(-1) for prm in tr.policy.parameters()]).cpu(),
                         _adam(one)[0], [torch.cat([st[k].reshape(-1).cpu() for st in tr.optimizer.state_dict()["state"].values()])
                                         for k in ("exp_avg", "exp_avg_sq")])
    out["vs_trainer_batch"] = ({k: one.last_batch[k].cpu() for k in tr.last_batch if k in one.last_batch},
                               {k: tr.last_batch[k].cpu() for k in tr.last_batch if k in one.last_batch})
    one.env.close()
    tr.env.close()
    # the evaluator: every rank returns the single-process results
    ev = PopulationEvaluator(PD, ND, seed=3, group=G)
    out["eval"] = [tuple(r) for r in ev.evaluate(pols, greedy=False)]
    # PBT: one ready event after the first iteration, decisions and post-event state the same on every rank
    pbt_pop = _dp_population(pols, first, c, G)
    single = PopulationEvaluator(PD, ND, seed=3)
    with pytest.raises(ValueError, match="group"):
        PopulationBasedTraining(pbt_pop, single, interval=1, fraction=0.5)
    single.close()
    pbt = PopulationBasedTraining(pbt_pop, ev, interval=1, fraction=0.5, seed=1)
    pbt.step()
    ev_hist = pbt.history[0]
    out["pbt"] = {"history": (ev_hist["fitness"], ev_hist["ranking"], ev_hist["copies"], ev_hist["factors"],
                              ev_hist["hyperparameters"]), "params": _params(pbt_pop), "adam": _adam(pbt_pop)}
    pbt_pop.env.close()
    ev.close()
    torch.save(out, os.path.join(outdir, "rank%d.pt" % rank))
    dist.barrier()
    dist.destroy_process_group()


def _check_two_ranks(backend, tmp_path):
    from wab_gym_b200 import PopulationEvaluator, VecEnv
    from wab_gym_b200.population import PPOPopulation
    outdir = str(tmp_path)
    pols = _pols()
    ref = PPOPopulation(VecEnv(PD * ND, seed=5, features=True), PD, HPS, policies=[copy.deepcopy(p) for p in pols], **KWD)
    ref.sample_seed = 4242
    ref.train_iteration()
    want_first = {k: ref.last_batch[k].cpu() for k in REC}
    ref.env.close()
    want_eval = PopulationEvaluator(PD, ND, seed=3).evaluate(pols, greedy=False)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, backend, outdir), nprocs=2, join=True)
    r = [torch.load(os.path.join(outdir, "rank%d.pt" % i), weights_only=False) for i in range(2)]
    # collection is world-size invariant: rank r's member p = columns [p n + first_r, ...) of the single process
    for rr in r:
        first, c = rr["first_c"]
        for k in REC:
            if k == "counters":
                assert torch.equal(rr["first"][k], want_first[k])
                continue
            for p in range(PD):
                assert torch.equal(rr["first"][k][:, p * c:(p + 1) * c], want_first[k][:, p * ND + first:p * ND + first + c]), k
    # bit-identical weights, Adam state and diagnostics on both ranks; resume from a per-rank state dict is bit-exact
    for key in ("params2", "params3", "params3_resumed"):
        assert all(torch.equal(a, b) for a, b in zip(r[0][key], r[1][key])), key
    assert all(torch.equal(x, y) for a, b in zip(r[0]["adam2"], r[1]["adam2"]) for x, y in zip(a, b))
    assert all(torch.equal(x, y) for x, y in zip(r[0]["params3"], r[0]["params3_resumed"]))
    for s0, s1 in zip(r[0]["stats"], r[1]["stats"]):
        assert torch.equal(s0["grad_norm"], s1["grad_norm"])
    # member p of the population = the 1-member data-parallel population on ids from p n
    for rr in r:
        c = rr["first_c"][1]
        for p in range(PD):
            m = rr["member%d" % p]
            assert torch.equal(rr["pop_batch2"]["counters"], m["batch"]["counters"])
            for k, v in m["batch"].items():
                if k == "counters":
                    continue
                got = rr["pop_batch2"][k][p * c:(p + 1) * c] if k == "bootstrap" else rr["pop_batch2"][k][:, p * c:(p + 1) * c]
                assert torch.equal(got, v), (p, k)
            for s_pop, s_one in zip(rr["stats"], m["stats"]):
                for k, v in s_one.items():
                    assert torch.equal(s_pop[k][p], v[0]), (p, k)
            assert torch.equal(rr["params2"][p], m["params"][0])
            assert all(torch.equal(x, y) for x, y in zip(rr["adam2"][p], m["adam"][0]))
        # a 1-member population at id 0 = PPOTrainer(group)
        a, b, pa, pb, aa, ab = rr["vs_trainer"]
        for sa, sb in zip(a, b):
            for k, v in sb.items():
                assert torch.equal(sa[k][0], v), k
        assert torch.equal(pa, pb) and all(torch.equal(x, y) for x, y in zip(aa, ab))
        ba, bb = rr["vs_trainer_batch"]
        assert all(torch.equal(ba[k], bb[k]) for k in bb)
    # the evaluator: every rank returns the single-process results bit for bit
    for rr in r:
        for got, want in zip(rr["eval"], want_eval):
            assert all(torch.equal(x, y) for x, y in zip(got, want))
    # PBT: the same decisions and post-event state on both ranks
    h0, h1 = r[0]["pbt"]["history"], r[1]["pbt"]["history"]
    assert torch.equal(h0[0], h1[0]) and h0[1:] == h1[1:] and len(h0[2]) == 1
    assert all(torch.equal(a, b) for a, b in zip(r[0]["pbt"]["params"], r[1]["pbt"]["params"]))
    assert all(torch.equal(x, y) for a, b in zip(r[0]["pbt"]["adam"], r[1]["pbt"]["adam"]) for x, y in zip(a, b))
    # the merged checkpoint resumes in one process: its next batch is the uninterrupted run's third
    merged = torch.load(os.path.join(outdir, "merged2.pt"), weights_only=False)
    one = PPOPopulation(VecEnv(PD * ND, seed=5, features=True), PD, HPS, policies=[copy.deepcopy(p) for p in pols], **KWD)
    one.load_state_dict(merged)
    one._collect()
    for k in REC:
        got = one.last_batch[k].cpu()
        if k == "counters":
            assert torch.equal(got, r[0]["third"][k])
            continue
        for rr in r:
            first, c = rr["first_c"]
            for p in range(PD):
                assert torch.equal(got[:, p * ND + first:p * ND + first + c], rr["third"][k][:, p * c:(p + 1) * c]), k
    one.env.close()


def test_two_ranks_on_one_gpu_over_gloo(tmp_path):
    _check_two_ranks("gloo", tmp_path)


def test_two_ranks_on_two_gpus_over_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL data-parallel populations need two visible GPUs; this machine shows %d" % torch.cuda.device_count())
    _check_two_ranks("nccl", tmp_path)
