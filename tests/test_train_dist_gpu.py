"""Data-parallel training on the GPU: policy draws keyed by global env id (a shard draws what the unsharded batch draws
for its rows), the deterministic cross-rank gradient sum, and PPOTrainer / A2CTrainer over two ranks (gloo on one GPU,
NCCL on two when the machine has them)."""
import ctypes
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

from tests.test_ppo_gpu import EPS, _check_parity, _materialise, _near_kinks, _perturbed, _record, _targets

pytestmark = pytest.mark.gpu


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _features(env, T):
    """T steps of real feature bytes [T, N, 28] under random actions."""
    g = torch.Generator(device="cuda").manual_seed(3)
    env.reset()
    out = torch.empty(T, env.num_envs, 28, dtype=torch.uint8, device="cuda")
    for t in range(T):
        out[t].copy_(env.last_features)
        env.step(torch.randint(0, env.n_actions, (env.num_envs,), device="cuda", generator=g).to(torch.uint8))
    return out


@pytest.mark.parametrize("noise", [0.01, 0.0])
@pytest.mark.parametrize("options", [None, {"lookout_only": False}, {"restrict_view": True}])
def test_shards_draw_what_the_unsharded_batch_draws(noise, options):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Affine1TC, Policy, PolicyTrainTC
    N, a, T, seed = 1100, 437, 3, 5                        # a: ragged, not a multiple of 4 (rows share sampling calls in fours)
    full = VecEnv(N, game_options=options, seed=seed, features=True)
    shards = [VecEnv(a, game_options=options, seed=seed, features=True, env_id_base=0),
              VecEnv(N - a, game_options=options, seed=seed, features=True, env_id_base=a)]
    spans = [(0, a), (a, N)]
    feats = _features(full, T)
    torch.manual_seed(1)
    pol = Policy(full.flat_dim, full.n_actions).cuda()
    tcs = [PolicyTrainTC(e, pol) for e in [full] + shards]
    ctr = torch.full((1,), 41, dtype=torch.int64, device="cuda")
    A, dim = full.n_actions, full.flat_dim

    def run(i, env, f):
        n, tc = f.shape[1], tcs[i]
        o = {"flat": env.flatten_features_noisy(f[0].contiguous(), torch.empty(n, dim, device="cuda"), noise, ctr),
             "h1": Affine1TC.__call__(tc, f[0].contiguous(), torch.empty(n, 128, device="cuda"), noise, ctr),
             "z3t": tc(f[0].contiguous(), torch.empty(n, 128, device="cuda"), noise, ctr)}
        acts, v, p, lp, z3 = (torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, device="cuda"),
                              torch.empty(n, A, device="cuda"), torch.empty(n, device="cuda"), torch.empty(n, 128, device="cuda"))
        tc.forward_sample(f[0].contiguous(), tc.heads, acts, value=v, probs=p, logp=lp, noise_scale=noise, counter=ctr, seed=77, z3=z3)
        o.update(actions=acts, value=v, probs=p, logp=lp, z3=z3)
        ctrs = torch.arange(50, 50 + T, dtype=torch.int64, device="cuda")
        act_t = torch.randint(0, A, (T, N), generator=torch.Generator(device="cuda").manual_seed(9), device="cuda").to(torch.uint8)
        lo, hi = (0, N) if i == 0 else spans[i - 1]
        act_t = act_t[:, lo:hi].contiguous()
        gl, gv = _targets(T, N, seed=4)
        gl, gv = gl[:, lo:hi].contiguous(), gv[:, lo:hi].contiguous()
        o["bwd_logp"], o["bwd_value"] = torch.empty(T, n, device="cuda"), torch.empty(T, n, device="cuda")
        tc.backward(f, ctrs, act_t, gl, gv, logp=o["bwd_logp"], value=o["bwd_value"], noise_scale=noise)
        o["ppo_logp"], o["ppo_value"], o["ppo_entropy"] = (torch.empty(T, n, device="cuda") for _ in range(3))
        tc.ppo_backward(f, ctrs, act_t, gl, gv, gl, None, None, EPS, 1e-3, 5e-4, 1e-4, logp=o["ppo_logp"],
                        value=o["ppo_value"], entropy=o["ppo_entropy"], noise_scale=noise)
        return o

    want = run(0, full, feats)
    for i, (env, (lo, hi)) in enumerate(zip(shards, spans), 1):
        got = run(i, env, feats[:, lo:hi].contiguous())
        for k, v in got.items():
            ref = want[k][:, lo:hi] if k.startswith(("bwd", "ppo")) else want[k][lo:hi]
            assert torch.equal(v, ref), (k, i)
    if noise:                                               # the second shard does not repeat the first one's draws
        other = run(2, shards[1], feats[:, :N - a].contiguous())
        assert not torch.equal(other["flat"], want["flat"][:N - a])
    for e in [full] + shards:
        e.close()


def test_one_rank_sum_of_the_fp64_gradient_is_the_fp32_gradient():
    T, n = 12, 1500
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=2)
    gl, gv = _targets(T, n)
    want = tc.backward(feats, ctrs, acts, gl, gv)
    got = tc.grad_sum_ranks(tc.grad_f64()[None].contiguous())
    assert torch.equal(got, want)
    want = tc.ppo_backward(feats, ctrs, acts, lp - 0.05, gl, gv, None, None, EPS, 1e-3, 5e-4, 1e-4)
    g64 = tc.grad_f64()
    assert torch.equal(tc.grad_sum_ranks(g64[None].contiguous()), want) and torch.equal(g64.float(), want)
    env.close()


@pytest.mark.parametrize("world", [1, 2, 8])
def test_sum_ranks_is_the_rank_order_fp64_sum(world):
    from wab_gym_b200 import _lib
    from wab_gym_b200.vec_env import _ptr
    lib = _lib.load()
    n, guard = 100003, 1024
    g = torch.Generator(device="cuda").manual_seed(world)
    x = torch.randn(world, n, dtype=torch.float64, device="cuda", generator=g) * \
        torch.exp2(torch.randint(-30, 30, (world, n), device="cuda", generator=g).double())
    buf = torch.full((n + 2 * guard,), 4321.0, device="cuda")
    assert lib.wab_policy_grad_sum_ranks(_ptr(x), world, n, _ptr(buf[guard:guard + n]), _stream()) == 0
    s = x[0].cpu().clone()
    for r in range(1, world):
        s += x[r].cpu()
    assert torch.equal(buf[guard:guard + n].cpu(), s.float())
    assert bool((buf[:guard] == 4321.0).all()) and bool((buf[-guard:] == 4321.0).all())


def test_grad_f64_and_sum_ranks_stay_in_bounds_and_refuse_bad_arguments():
    from wab_gym_b200.vec_env import _ptr
    T, n = 4, 700
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=6)
    gl, gv = _targets(T, n)
    want = tc.backward(feats, ctrs, acts, gl, gv)
    guard = 512
    buf = torch.full((tc.n_params + 2 * guard,), -9.0, dtype=torch.float64, device="cuda")
    got = tc.grad_f64(buf[guard:guard + tc.n_params])
    torch.cuda.synchronize()
    assert torch.equal(got.float(), want)
    assert bool((buf[:guard] == -9.0).all()) and bool((buf[-guard:] == -9.0).all())
    lib, s, A = tc.lib, tc.scratch, tc.heads[0].shape[0] - 1
    out64 = torch.empty(tc.n_params + 1, dtype=torch.float64, device="cuda")
    out32 = torch.empty(tc.n_params + 1, device="cuda")
    f64 = lib.wab_policy_backward_grad_f64
    assert f64(env._h, _ptr(s), s.numel(), A, _ptr(out64), _stream()) == 0
    assert f64(None, _ptr(s), s.numel(), A, _ptr(out64), _stream()) == 1
    assert f64(env._h, None, s.numel(), A, _ptr(out64), _stream()) == 1
    assert f64(env._h, _ptr(s), s.numel(), A, None, _stream()) == 1
    assert f64(env._h, _ptr(s), s.numel() - 1, A, _ptr(out64), _stream()) == 2
    assert f64(env._h, ctypes.c_void_p(s.data_ptr() + 8), s.numel(), A, _ptr(out64), _stream()) == 2
    assert f64(env._h, _ptr(s), s.numel(), A, ctypes.c_void_p(out64.data_ptr() + 4), _stream()) == 2
    assert f64(env._h, _ptr(s), s.numel(), 9, _ptr(out64), _stream()) == 3
    sr = lib.wab_policy_grad_sum_ranks
    assert sr(_ptr(out64), 1, 16, _ptr(out32), _stream()) == 0
    assert sr(None, 1, 16, _ptr(out32), _stream()) == 1 and sr(_ptr(out64), 1, 16, None, _stream()) == 1
    assert sr(_ptr(out64), 0, 16, _ptr(out32), _stream()) == 2 and sr(_ptr(out64), 1, -1, _ptr(out32), _stream()) == 2
    assert sr(ctypes.c_void_p(out64.data_ptr() + 4), 1, 16, _ptr(out32), _stream()) == 2
    assert sr(_ptr(out64), 1, 16, ctypes.c_void_p(out32.data_ptr() + 2), _stream()) == 2
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        tc.grad_sum_ranks(out64[:tc.n_params][None].float())
    env.close()


def test_sharded_ppo_gradient_meets_the_parity_rule():
    """Each shard's ppo_backward on its rows with the global count's weights, grad_f64, sum_ranks: the same parity rule
    against fp64 autograd of ppo_loss as the single-handle gradient over the same rows."""
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import PolicyTrainTC
    T, n, a = 24, 4099, 1999                # test_ppo_gpu's ragged case (its perturbation clips rows on both sides), two shards
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, head_scale=1.0)
    adv, target = _targets(T, n, seed=5)
    x = _materialise(env, feats, ctrs, 0.01)
    new, r = _perturbed(pol, x, acts, lp, adv)
    bad = _near_kinks(new, x) | ((r - (1 + EPS)).abs() < 1e-3) | ((r - (1 - EPS)).abs() < 1e-3)
    sel = torch.nonzero(~bad).squeeze(1)
    m = sel.numel()
    w = (1.0 / m, 0.5 / m, 0.01 / m)
    rlp, rv = torch.empty_like(lp), torch.empty_like(lp)
    one = PolicyTrainTC(env, new)
    single = one.ppo_backward(feats, ctrs, acts, lp, adv, target, sel.to(torch.int32),
                              torch.tensor([m], dtype=torch.int64, device="cuda"), EPS, *w, logp=rlp, value=rv)
    _check_parity(new, single, (x, acts, lp, adv, target, sel, w, (rlp, rv)))
    parts = []
    for lo, hi in ((0, a), (a, n)):
        sh = VecEnv(hi - lo, seed=1, features=True, env_id_base=lo)
        tc_s = PolicyTrainTC(sh, new)
        t, j = sel // n, sel % n
        mine = (j >= lo) & (j < hi)
        rows = (t[mine] * (hi - lo) + j[mine] - lo).to(torch.int32)
        sl = lambda z: z[:, lo:hi].contiguous()
        slp, sv = torch.empty(T, hi - lo, device="cuda"), torch.empty(T, hi - lo, device="cuda")
        tc_s.ppo_backward(sl(feats), ctrs, sl(acts), sl(lp), sl(adv), sl(target), rows,
                          torch.tensor([rows.numel()], dtype=torch.int64, device="cuda"), EPS, *w, logp=slp, value=sv)
        parts.append(tc_s.grad_f64())
        assert torch.equal(slp.reshape(-1)[rows.long()], rlp[:, lo:hi].reshape(-1)[rows.long()])
        sh.close()
    sharded = one.grad_sum_ranks(torch.stack(parts))
    _check_parity(new, sharded, (x, acts, lp, adv, target, sel, w, (rlp, rv)))
    env.close()


# ---- two ranks ------------------------------------------------------------------------------------------------------

N_TOTAL, T_H, SEED = 1001, 8, 11          # ragged shards: 501 + 500


def _flat_params(tr):
    return torch.cat([p.detach().reshape(-1) for p in tr.policy.parameters()]).cpu()


def _make(kind, n, first, group=None, horizon=None, **kw):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    env = VecEnv(n, seed=SEED, features=True, emit_grids=False, env_id_base=first, device=torch.device("cuda", torch.cuda.current_device()))
    torch.manual_seed(0)
    pol = Policy(env.flat_dim, env.n_actions)
    if kind == "ppo":
        return PPOTrainer(env, pol, horizon=horizon or T_H, group=group, **kw)
    return A2CTrainer(env, pol, horizon=horizon, mode=kind, tensor_cores=True, lr=3e-3, group=group, **kw)


REC_KEYS = ("features", "counters", "actions", "logp", "value", "reward", "done")


def _record_of(tr):
    return {k: tr.last_batch[k].cpu().clone() for k in REC_KEYS}


def _worker(rank, world, port, backend, outdir):
    import torch.distributed as dist
    from wab_gym_b200.sharding import merge_trainer_state_dicts, shard_range
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=world)
    first, count = shard_range(N_TOTAL, rank, world)
    out = {}
    # first iteration: the collected record, advantages, targets and the (unclipped) gradient
    tr = _make("ppo", count, first, dist.group.WORLD, epochs=1, minibatches=1, max_grad_norm=float("inf"))
    info = tr.train_iteration()
    out["first"] = _record_of(tr)
    out["first_adv"], out["first_target"] = tr.last_batch["advantage"].cpu(), tr.last_batch["target"].cpu()
    out["first_grad"] = torch.cat([p.grad.reshape(-1) for p in tr.policy.parameters()]).cpu()
    out["first_norm"] = info["grad_norm"].cpu()
    tr.env.close()
    # three PPO iterations, twice; a checkpoint after two, resumed on the same layout
    runs = []
    for again in range(2):
        tr = _make("ppo", count, first, dist.group.WORLD, epochs=2, minibatches=3)
        for it in range(3):
            if it == 2 and again == 0:
                sds = [None] * world
                dist.all_gather_object(sds, tr.state_dict())
                merged = merge_trainer_state_dicts(sds)
                if rank == 0:
                    torch.save(merged, os.path.join(outdir, "ppo_sd2.pt"))
            tr.train_iteration()
        runs.append(_flat_params(tr))
        if again == 0:
            out["third"] = _record_of(tr)
        tr.env.close()
    out["ppo_params"], out["ppo_params_again"] = runs
    res = _make("ppo", count, first, dist.group.WORLD, epochs=2, minibatches=3)
    res.train_iteration()                                       # a state of its own first
    res.load_state_dict(merged)
    res.train_iteration()
    out["ppo_params_resumed"] = _flat_params(res)
    res.env.close()
    # a single-process checkpoint (written by the test before spawning) resumed on two ranks: the next collected batch
    single = torch.load(os.path.join(outdir, "single_sd2.pt"), weights_only=False)
    tr = _make("ppo", count, first, dist.group.WORLD, epochs=2, minibatches=3)
    tr.load_state_dict(single)
    tr._collect_tc()
    out["from_single"] = _record_of(tr)
    tr.env.close()
    for mode in ("episodic", "horizon"):
        tr = _make(mode, count, first, dist.group.WORLD, **({"horizon": 16} if mode == "horizon" else {}))
        for _ in range(3):
            tr.train_iteration()
        out["a2c_" + mode] = _flat_params(tr)
        tr.env.close()
    torch.save(out, os.path.join(outdir, "rank%d.pt" % rank))
    dist.barrier()
    dist.destroy_process_group()


def _single_process_reference(outdir):
    """The same runs in one process over all N_TOTAL envs; writes the checkpoint after two iterations."""
    ref = {}
    tr = _make("ppo", N_TOTAL, 0, epochs=1, minibatches=1, max_grad_norm=float("inf"))
    tr.train_iteration()
    ref["first"] = _record_of(tr)
    ref["first_adv"], ref["first_target"] = tr.last_batch["advantage"].cpu(), tr.last_batch["target"].cpu()
    ref["first_grad"] = torch.cat([p.grad.reshape(-1) for p in tr.policy.parameters()]).cpu()
    tr.env.close()
    tr = _make("ppo", N_TOTAL, 0, epochs=2, minibatches=3)
    for it in range(3):
        if it == 2:
            torch.save(tr.state_dict(), os.path.join(outdir, "single_sd2.pt"))
        tr.train_iteration()
    ref["third"] = _record_of(tr)
    tr.env.close()
    return ref


def _check_two_ranks(backend, tmp_path):
    outdir = str(tmp_path)
    ref = _single_process_reference(outdir)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, backend, outdir), nprocs=2, join=True)
    r0, r1 = (torch.load(os.path.join(outdir, "rank%d.pt" % r), weights_only=False) for r in range(2))
    # collection is invariant to the world size: the first batch (same weights), and the batch after a single-process
    # checkpoint (the runs' weights differ after training: training is not bit-exact across world sizes)
    for k in REC_KEYS:
        for rec, want in (("first", ref["first"][k]), ("from_single", ref["third"][k])):
            got = torch.cat([r0[rec][k], r1[rec][k]], dim=1) if k != "counters" else r0[rec][k]
            assert torch.equal(got, want), (rec, k)
            assert k != "counters" or torch.equal(r1[rec][k], want), (rec, k)
    assert torch.equal(torch.cat([r0["first_target"], r1["first_target"]], 1), ref["first_target"])   # GAE is per env
    adv = torch.cat([r0["first_adv"], r1["first_adv"]], 1)
    assert torch.allclose(adv, ref["first_adv"], rtol=1e-5, atol=1e-5)
    # the first gradient: the same on both ranks, and the single process's within the replay bound of test_ppo_gpu
    assert torch.equal(r0["first_grad"], r1["first_grad"]) and torch.equal(r0["first_norm"], r1["first_norm"])
    g, want = r0["first_grad"], ref["first_grad"]
    assert torch.allclose(g, want, rtol=1e-5, atol=1e-5 * float(want.abs().max()))
    for k in ("ppo_params", "ppo_params_again", "ppo_params_resumed", "a2c_episodic", "a2c_horizon"):
        assert torch.equal(r0[k], r1[k]), k                     # bit-identical weights on every rank
    assert torch.equal(r0["ppo_params"], r0["ppo_params_again"])          # two runs are identical
    assert torch.equal(r0["ppo_params"], r0["ppo_params_resumed"])        # a 2-rank resume is bit-exact
    # a 2-rank checkpoint in a single process: its next collected batch is the uninterrupted run's
    merged = torch.load(os.path.join(outdir, "ppo_sd2.pt"), weights_only=False)
    tr = _make("ppo", N_TOTAL, 0, epochs=2, minibatches=3)
    tr.load_state_dict(merged)
    tr._collect_tc()
    for k in REC_KEYS:
        want = torch.cat([r0["third"][k], r1["third"][k]], 1) if k != "counters" else r0["third"][k]
        assert torch.equal(tr.last_batch[k].cpu(), want), k
    tr.env.close()


def test_two_ranks_on_one_gpu_over_gloo(tmp_path):
    _check_two_ranks("gloo", tmp_path)


def test_two_ranks_on_two_gpus_over_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL data-parallel training needs two visible GPUs; this machine shows %d" % torch.cuda.device_count())
    _check_two_ranks("nccl", tmp_path)


def test_a_group_of_one_rank_is_the_single_process_path():
    import torch.distributed as dist
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        # a group of one rank: the single-process path, bit for bit
        a, b = _make("ppo", 600, 0, dist.group.WORLD, epochs=1, minibatches=2), _make("ppo", 600, 0, None, epochs=1, minibatches=2)
        assert a.group is None
        a.train_iteration(); b.train_iteration()
        assert torch.equal(_flat_params(a), _flat_params(b))
        a.env.close(); b.env.close()
    finally:
        dist.destroy_process_group()


def _refusal_worker(rank, world, port, outdir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    res = []
    for case in ("gap", "hyper", "torch_path"):
        first, count = (0, 300) if rank == 0 else ((301 if case == "gap" else 300), 300)
        try:
            if case == "torch_path":
                env = VecEnv(count, seed=SEED, features=True, env_id_base=first)
                A2CTrainer(env, group=dist.group.WORLD)
            else:
                _make("ppo", count, first, dist.group.WORLD, epochs=1, minibatches=2 + (rank if case == "hyper" else 0))
            res.append("accepted")
        except ValueError:
            res.append("refused")
    torch.save(res, os.path.join(outdir, "refusal%d.pt" % rank))
    dist.destroy_process_group()


def test_two_ranks_refuse_bad_layouts_on_every_rank(tmp_path):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_refusal_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        assert torch.load(os.path.join(str(tmp_path), "refusal%d.pt" % r)) == ["refused"] * 3


def _memory_worker(rank, world, port, outdir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from wab_gym_b200.sharding import shard_range
    first, count = shard_range(2 * 32768, rank, world)
    tr = _make("ppo", count, first, dist.group.WORLD, horizon=64)
    torch.save(_peak(tr), os.path.join(outdir, "peak%d.pt" % rank))
    tr.env.close()
    dist.destroy_process_group()


def _peak(tr):
    tr.train_iteration()                                       # the first iteration allocates Adam's state
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    tr.train_iteration()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def test_rank_memory_is_the_single_process_peak_plus_the_gather_buffer(tmp_path):
    tr = _make("ppo", 32768, 0, horizon=64)
    single = _peak(tr)
    n_params = tr._tc.n_params
    tr.env.close()
    del tr
    torch.cuda.empty_cache()
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_memory_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        peak = torch.load(os.path.join(str(tmp_path), "peak%d.pt" % r))
        assert peak <= single + 2 * n_params * 8 + 16 * 2 ** 20, (peak, single)
