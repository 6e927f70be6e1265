"""Training on the tensor cores: the backward pass of Policy.forward (``wab_policy_backward``) against fp64 autograd
through ``Policy`` on the materialised input, and ``A2CTrainer(tensor_cores=True)`` against the torch trainer."""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _record(n, T, noise, seed=1, options=None, scale=3.0):
    """A real rollout through forward_sample: features [T, N, 28], counters [T], actions, logp, value."""
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy, PolicyTrainTC
    env = VecEnv(n, game_options=options, seed=seed, features=True)
    env.reset()
    torch.manual_seed(seed)
    pol = Policy(env.flat_dim, env.n_actions).cuda()
    with torch.no_grad():                                # both leaky branches well populated
        for lin in (pol.affine1, pol.affine2, pol.affine3):
            lin.weight.mul_(scale)
        pol.affine3.bias[:32] += 3.5                     # a quarter of the units straddle the upper clamp at +4 (the lower
        pol.action_head.weight.mul_(4.0)                 # one, leaky(z3) < -4, needs z3 < -400: out of reach of any policy here)
    tc = PolicyTrainTC(env, pol)
    feats = torch.empty(T, n, 28, dtype=torch.uint8, device="cuda")
    ctrs = torch.empty(T, dtype=torch.int64, device="cuda")
    acts = torch.empty(T, n, dtype=torch.uint8, device="cuda")
    lp, v = torch.empty(T, n, device="cuda"), torch.empty(T, n, device="cuda")
    ctr = torch.full((1,), 100, dtype=torch.int64, device="cuda")
    for t in range(T):
        ctr += 1
        feats[t].copy_(env.last_features)
        ctrs[t:t + 1].copy_(ctr)
        tc.forward_sample(feats[t], tc.heads, acts[t], value=v[t], logp=lp[t], noise_scale=noise, counter=ctr, seed=17)
        env.step(acts[t])
    return env, pol, tc, feats, ctrs, acts, lp, v


def _upstream(T, n, seed=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    gl = torch.randn(T, n, device="cuda", generator=g)
    gv = torch.randn(T, n, device="cuda", generator=g)
    gl[T // 3:T // 2] = 0.0                              # a block of rows without upstream gradient
    gv[T // 3:T // 2] = 0.0
    return gl, gv


def _materialise(env, feats, ctrs, noise):
    """The policy input each step saw: flatten_features_noisy per step under that step's counter, f32[T, N, flat_dim]."""
    T, n = feats.shape[:2]
    flat = torch.empty(T, n, env.flat_dim, device="cuda")
    step = torch.empty(n, env.flat_dim, device="cuda")                 # 16-byte aligned for any N
    for t in range(T):
        flat[t].copy_(env.flatten_features_noisy(feats[t], step, noise, ctrs[t:t + 1]))
    return flat


def _torch_grads(env, pol, feats, ctrs, acts, gl, gv, noise, dtype):
    """Autograd through Policy on the input materialised with flatten_features_noisy per step and counter."""
    T, n = acts.shape
    p = copy.deepcopy(pol).to(dtype)
    flat = _materialise(env, feats, ctrs, noise)
    probs, value = p(flat.to(dtype).reshape(T * n, -1))
    logp = torch.log(probs.gather(1, acts.reshape(-1, 1).long()).squeeze(1))
    loss = (gl.reshape(-1).to(dtype) * logp).sum() + (gv.reshape(-1).to(dtype) * value.squeeze(1)).sum()
    return torch.autograd.grad(loss, list(p.parameters()))


def _off_kinks(env, pol, feats, ctrs, gl, gv, noise, rel=3e-5):
    """The upstream gradients with rows zeroed whose fp64 pre-activations lie within `rel` of their layer's largest
    magnitude from a kink (leaky-ReLU at 0, the clamp at +-4): there an fp32 forward — torch's or the library's — may
    take the other branch, and the gradient of that row changes by O(1). Both sides get the same zeroed rows."""
    T, n = gl.shape
    flat = _materialise(env, feats, ctrs, noise)
    p = copy.deepcopy(pol).double()
    with torch.no_grad():
        z1 = p.affine1(flat.reshape(T * n, -1).double())
        z2 = p.affine2(F.leaky_relu(z1))
        z3 = p.affine3(F.leaky_relu(z2))
        y = F.leaky_relu(z3)
        near = torch.zeros(T * n, dtype=torch.bool, device="cuda")
        for z, k in ((z1, 0.0), (z2, 0.0), (z3, 0.0), (y, 4.0), (y, -4.0)):
            near |= ((z - k).abs() < rel * float(z.abs().max())).any(1)
    keep = (~near).view(T, n).float()
    _off_kinks.clamped = float(((y > 4.0).any(1) & ~near).float().mean())     # rows whose gradient passes the clamp mask
    return (gl * keep).contiguous(), (gv * keep).contiguous(), float(near.float().mean())


def _check_parity(pol, lib_flat, env, feats, ctrs, acts, gl, gv, noise):
    g64 = _torch_grads(env, pol, feats, ctrs, acts, gl, gv, noise, torch.float64)
    g32 = _torch_grads(env, pol, feats, ctrs, acts, gl, gv, noise, torch.float32)
    off, report, ok = 0, [], True
    for (name, prm), w64, w32 in zip(pol.named_parameters(), g64, g32):
        got = lib_flat[off:off + prm.numel()].view_as(prm).double()
        off += prm.numel()
        err, err32, big = float((got - w64).abs().max()), float((w32.double() - w64).abs().max()), float(w64.abs().max())
        ok &= err <= 2 * err32 + 1e-6 * big
        report.append("%s: library error %.3g, torch fp32 error %.3g, largest %.3g" % (name, err, err32, big))
    assert off == lib_flat.numel()
    print("\n".join(report))
    assert ok, "\n".join(report)


@pytest.mark.parametrize("n,noise,options", [
    (1000, 0.0, None), (4099, 0.01, None), (1000, 0.01, {"lookout_only": False}), (1000, 0.01, {"restrict_view": True}),
])
def test_backward_matches_fp64_autograd(n, noise, options):
    T = 40
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, options=options)
    gl, gv, frac = _off_kinks(env, pol, feats, ctrs, *_upstream(T, n), noise)
    assert frac < 0.2 and _off_kinks.clamped > 0.05, (frac, _off_kinks.clamped)
    rlp, rv = torch.full_like(lp, float("nan")), torch.full_like(v, float("nan"))
    grad = tc.backward(feats, ctrs, acts, gl, gv, noise_scale=noise, logp=rlp, value=rv)
    assert torch.isfinite(grad).all()
    assert torch.equal(rlp, lp) and torch.equal(rv, v)           # the recomputed forward is the rollout's, bit for bit
    _check_parity(pol, grad, env, feats, ctrs, acts, gl, gv, noise)
    env.close()


def test_backward_is_deterministic_and_skipping_rows_is_free():
    T, n = 24, 3000
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=4)
    gl, gv, _ = _off_kinks(env, pol, feats, ctrs, *_upstream(T, n, seed=5), 0.01)
    a = tc.backward(feats, ctrs, acts, gl, gv)
    b = tc.backward(feats, ctrs, acts, gl, gv)
    assert torch.equal(a, b)                                      # fixed-order reductions: bit-identical
    active = ((gl != 0) | (gv != 0)).reshape(-1)
    rows = torch.nonzero(active).squeeze(1).to(torch.int32)
    pad = torch.full((T * n - rows.numel(),), -7, dtype=torch.int32, device="cuda")   # never read: beyond the count
    n_rows = torch.tensor([rows.numel()], dtype=torch.int64, device="cuda")
    c = tc.backward(feats, ctrs, acts, gl, gv, rows=torch.cat([rows, pad]), n_rows=n_rows)
    _check_parity(pol, c, env, feats, ctrs, acts, gl, gv, 0.01)
    assert torch.equal(c, tc.backward(feats, ctrs, acts, gl, gv, rows=torch.cat([rows, pad]), n_rows=n_rows))
    zero = tc.backward(feats, ctrs, acts, gl, gv, rows=rows, n_rows=torch.zeros(1, dtype=torch.int64, device="cuda"))
    assert torch.equal(zero, torch.zeros_like(zero))
    env.close()


def test_backward_stays_inside_its_buffers():
    T, n = 8, 1500
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=6)
    gl, gv = _upstream(T, n, seed=7)
    want = tc.backward(feats, ctrs, acts, gl, gv)
    guard = 4096
    gbuf = torch.full((tc.n_params + 2 * guard,), 12345.0, device="cuda")
    sbuf = torch.full((tc.scratch.numel() + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
    tc.scratch = sbuf[guard:guard + tc.scratch.numel()]
    got = tc.backward(feats, ctrs, acts, gl, gv, out=gbuf[guard:guard + tc.n_params])
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert bool((gbuf[:guard] == 12345.0).all()) and bool((gbuf[-guard:] == 12345.0).all())
    assert bool((sbuf[:guard] == 0xA5).all()) and bool((sbuf[-guard:] == 0xA5).all())
    env.close()


def _trainers(n, mode, seed=2, T=None):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.policy import Policy
    env = VecEnv(n, seed=seed, features=True, emit_grids=False)
    torch.manual_seed(seed)
    pol = Policy(env.flat_dim, env.n_actions).cuda()
    return A2CTrainer(env, pol, mode=mode, tensor_cores=True, horizon=T)


def _backward_with(policy, tr, rec, gl, gv):
    """wab_policy_backward of the recorded batch under the weights of `policy` (the trainer's before its Adam step)."""
    from wab_gym_b200.policy import PolicyTrainTC
    tc = PolicyTrainTC(tr.env, policy)
    return tc.backward(rec["features"], rec["counters"], rec["actions"], gl.contiguous(), gv.contiguous())


@pytest.mark.parametrize("mode", ["episodic", "horizon"])
def test_trainer_gradients_match_torch_replay(mode):
    """One iteration: the loss and gradients of the tensor-core trainer equal the torch reference replayed on the recorded
    actions and materialised inputs, within the tolerance of the parity test."""
    tr = _trainers(2000, mode, T=40 if mode == "horizon" else None)
    before = copy.deepcopy(tr.policy)
    info = tr.train_iteration()
    rec = tr.last_batch
    env, T, n = tr.env, rec["actions"].shape[0], tr.env.num_envs
    flat = _materialise(env, rec["features"], rec["counters"], 0.01)
    probs, value = before(flat.reshape(T * n, -1))
    logp = torch.log(probs.gather(1, rec["actions"].reshape(-1, 1).long()).squeeze(1)).view(T, n)
    assert torch.allclose(logp, rec["logp"], rtol=1e-5, atol=1e-5) and torch.allclose(value.squeeze(1).view(T, n), rec["value"], rtol=1e-5, atol=1e-5)
    g_logp, g_value = rec["g_logp"], rec["g_value"]
    assert torch.isfinite(info["loss"]) and float((g_logp != 0).float().mean()) > 0.1
    from wab_gym_b200.a2c import episodic_actor_critic_loss, horizon_actor_critic_loss
    value = value.squeeze(1).view(T, n)                  # the loss of the torch trainer on the replayed tensors
    if mode == "episodic":
        want, _ = episodic_actor_critic_loss(logp, value, rec["reward"], rec["done"], tr.gamma, tr.eps)
    else:                                                # the bootstrap: the last observation under the last counter
        boot = env.flatten_features_noisy(env.last_features, torch.empty(n, env.flat_dim, device="cuda"), 0.01, tr._ctr)
        want, _ = horizon_actor_critic_loss(logp, value, rec["reward"], rec["done"], before(boot)[1].squeeze(1).detach(), tr.gamma, tr.eps)
    assert torch.allclose(info["loss"], want.detach(), rtol=1e-4, atol=1e-3), (float(info["loss"]), float(want))
    # the trainer's gradient is the library backward of the recorded batch (here over every row, without the compaction)
    grad = torch.cat([p.grad.reshape(-1) for p in tr.policy.parameters()])
    full = _backward_with(before, tr, rec, g_logp, g_value)
    assert torch.allclose(grad, full, rtol=1e-5, atol=1e-5 * float(full.abs().max()))
    gl, gv, _ = _off_kinks(env, before, rec["features"], rec["counters"], g_logp, g_value, 0.01)
    _check_parity(before, _backward_with(before, tr, rec, gl, gv), env, rec["features"], rec["counters"], rec["actions"], gl, gv, 0.01)
    env.close()


@pytest.mark.parametrize("mode", ["episodic", "horizon"])
def test_trainer_runs_and_resumes_bit_exactly(mode):
    n, iters = 1024, 3
    T = 30 if mode == "horizon" else None
    a = _trainers(n, mode, T=T)
    p0 = [p.detach().clone() for p in a.policy.parameters()]
    a.env.stats(clear=True)
    for _ in range(iters):
        info = a.train_iteration()
        assert torch.isfinite(info["loss"])
    st = a.env.stats()
    assert st["steps"] == n * a.horizon * iters and st["bad_actions"] == 0
    assert any(not torch.equal(p, q) for p, q in zip(p0, a.policy.parameters()))
    b = _trainers(n, mode, T=T)
    for _ in range(2):
        b.train_iteration()
    sd = b.state_dict()
    b.env.close()
    c = _trainers(n, mode, T=T)
    c.train_iteration()                                      # a state of its own first: everything comes from the state dict
    c.load_state_dict(sd)
    c.train_iteration()
    for p, q in zip(a.policy.parameters(), c.policy.parameters()):
        assert torch.equal(p, q)
    a.env.close(); c.env.close()


def test_trainer_refuses_what_the_kernels_do_not_cover():
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.policy import Policy
    env = VecEnv(256, seed=1, features=True)
    with pytest.raises(ValueError):
        A2CTrainer(env, Policy(env.flat_dim, env.n_actions).double(), tensor_cores=True)
    bad = Policy(env.flat_dim, env.n_actions)
    bad.affine2 = torch.nn.Linear(128, 140)
    with pytest.raises(ValueError):
        A2CTrainer(env, bad, tensor_cores=True)
    env.close()
    with pytest.raises(ValueError):
        A2CTrainer(VecEnv(256, seed=1), tensor_cores=True)


def test_tensor_core_training_needs_a_tenth_of_the_memory():
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.policy import Policy
    peaks = {}
    for tc in (False, True):
        env = VecEnv(32768, seed=3, features=True, emit_grids=False)
        torch.manual_seed(0)
        tr = A2CTrainer(env, Policy(env.flat_dim, env.n_actions), tensor_cores=tc)
        tr.train_iteration()                                   # the first iteration allocates Adam's state
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        tr.train_iteration()
        torch.cuda.synchronize()
        peaks[tc] = torch.cuda.max_memory_allocated() - base
        env.close()
        del tr, env
        torch.cuda.empty_cache()
    assert peaks[True] * 10 <= peaks[False], peaks
