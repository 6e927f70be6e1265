"""PPO on the tensor cores: ``wab_policy_ppo_backward`` against the existing backward pass and against fp64 autograd of
``ppo_loss`` through ``Policy`` on the materialised input, and ``PPOTrainer`` against a torch replay of its batch."""
import copy
import ctypes

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

EPS = 0.2


def _record(n, T, noise, seed=1, options=None, scale=3.0, head_scale=4.0):
    """A real rollout through forward_sample: env, policy, its PolicyTrainTC, features [T, N, 28], counters [T], actions,
    logp, value."""
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy, PolicyTrainTC
    env = VecEnv(n, game_options=options, seed=seed, features=True)
    env.reset()
    torch.manual_seed(seed)
    pol = Policy(env.flat_dim, env.n_actions).cuda()
    with torch.no_grad():                                # both leaky branches and the upper clamp populated
        for lin in (pol.affine1, pol.affine2, pol.affine3):
            lin.weight.mul_(scale)
        pol.affine3.bias[:32] += 3.5
        pol.action_head.weight.mul_(head_scale)
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


def _materialise(env, feats, ctrs, noise):
    """The policy input each step saw, f32[T N, flat_dim]."""
    T, n = feats.shape[:2]
    flat = torch.empty(T, n, env.flat_dim, device="cuda")
    step = torch.empty(n, env.flat_dim, device="cuda")
    for t in range(T):
        flat[t].copy_(env.flatten_features_noisy(feats[t], step, noise, ctrs[t:t + 1]))
    return flat.reshape(T * n, -1)


def _heads(pol, x):
    """log pi(. | x), V(x) and the entropy through Policy's layers (log-softmax of the logits, so no log 0)."""
    h = F.leaky_relu(pol.affine1(x))
    h = F.leaky_relu(pol.affine2(h))
    h = torch.clamp(F.leaky_relu(pol.affine3(h)), -4, 4)
    logq = torch.log_softmax(pol.action_head(h), -1)
    return logq, pol.value_head(h).squeeze(1), -(logq.exp() * logq).sum(-1)


def _near_kinks(pol, x, rel=3e-5):
    """Rows whose fp64 pre-activations lie within `rel` of their layer's largest magnitude from a kink (leaky-ReLU at 0,
    the clamp at +-4): there any fp32 forward may take the other branch."""
    p = copy.deepcopy(pol).double()
    with torch.no_grad():
        z1 = p.affine1(x.double())
        z2 = p.affine2(F.leaky_relu(z1))
        z3 = p.affine3(F.leaky_relu(z2))
        y = F.leaky_relu(z3)
        near = torch.zeros(x.shape[0], dtype=torch.bool, device="cuda")
        for z, k in ((z1, 0.0), (z2, 0.0), (z3, 0.0), (y, 4.0), (y, -4.0)):
            near |= ((z - k).abs() < rel * float(z.abs().max())).any(1)
    return near


def _ppo_grads(pol, x, acts, logp_old, adv, target, sel, w, at, dtype):
    """Autograd of sum over rows `sel` of the per-row objective (weights w = (w_pi, w_v, w_H)) through Policy. With `at`
    = (logp, value) f32[T, N], log pi(a | x) and V(x) take those values (the gradient still flows through Policy)."""
    from wab_gym_b200.ppo import ppo_loss
    p = copy.deepcopy(pol).to(dtype)
    logq, value, ent = _heads(p, x[sel].to(dtype))
    logp = logq.gather(1, acts.reshape(-1)[sel].long()[:, None]).squeeze(1)
    if at is not None:
        logp = logp + (at[0].reshape(-1)[sel].to(dtype) - logp).detach()
        value = value + (at[1].reshape(-1)[sel].to(dtype) - value).detach()
    m = sel.numel()
    loss, _ = ppo_loss(logp, value, ent, logp_old.reshape(-1)[sel].to(dtype), adv.reshape(-1)[sel].to(dtype),
                       target.reshape(-1)[sel].to(dtype), EPS, w[1] / w[0], w[2] / w[0])
    return torch.autograd.grad(loss * (m * w[0]), list(p.parameters()))


def _check_parity(pol, lib_flat, args):
    if len(args) == 7:
        args = (*args, None)
    g64, g32 = _ppo_grads(pol, *args, torch.float64), _ppo_grads(pol, *args, torch.float32)
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


def _targets(T, n, seed=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(T, n, device="cuda", generator=g), torch.randn(T, n, device="cuda", generator=g)


def test_reduces_to_the_existing_backward_on_the_recording_weights():
    T, n = 24, 2000
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=2)
    adv, target = _targets(T, n)
    w_pi, w_v = 0.25, 0.5                               # exact in fp32: -w_pi A and w_v (V - R) round as the kernel's
    rlp, rv, ent = (torch.full_like(lp, float("nan")) for _ in range(3))
    got = tc.ppo_backward(feats, ctrs, acts, lp, adv, target, None, None, float("inf"), w_pi, w_v, 0.0, logp=rlp, value=rv,
                          entropy=ent)
    want = tc.backward(feats, ctrs, acts, (-w_pi * adv).contiguous(), (w_v * (v - target)).contiguous())
    assert torch.equal(got, want)
    assert torch.equal(rlp, lp) and torch.equal(rv, v)  # r = exp(0) = 1 bit for bit
    logq, _, ent64 = _heads(copy.deepcopy(pol).double(), _materialise(env, feats, ctrs, 0.01).double())
    assert torch.allclose(ent.double().reshape(-1), ent64, rtol=1e-5, atol=1e-5)
    env.close()


def _perturbed(pol, x, acts, logp_old, adv):
    """A copy of `pol` moved so that the ratios spread past both clip bounds: a small relative change everywhere plus a
    change of the action head, scaled up until at least 5 % of the rows are clipped on each side (fp64)."""
    g = torch.Generator(device="cuda").manual_seed(11)
    for c in (0.02, 0.05, 0.1, 0.2, 0.5, 1.0, 2.0):
        p = copy.deepcopy(pol)
        with torch.no_grad():
            for prm in p.parameters():
                prm.add_(1e-3 * prm.abs().mean() * torch.randn(prm.shape, device="cuda", generator=g))
            p.action_head.weight.add_(c * torch.randn(p.action_head.weight.shape, device="cuda", generator=g))
            logq, _, _ = _heads(copy.deepcopy(p).double(), x.double())
            r = torch.exp(logq.gather(1, acts.reshape(-1, 1).long()).squeeze(1) - logp_old.reshape(-1).double())
        a = adv.reshape(-1)
        above, below = float(((a > 0) & (r > 1 + EPS)).float().mean()), float(((a < 0) & (r < 1 - EPS)).float().mean())
        if above > 0.05 and below > 0.05:
            return p, r
    raise AssertionError("no perturbation spreads the ratios past both bounds")


@pytest.mark.parametrize("n,noise,options,w_h", [
    (1000, 0.0, None, 0.0), (4099, 0.01, None, 0.02), (1000, 0.01, {"lookout_only": False}, 0.02),
    (1000, 0.01, {"restrict_view": True}, 0.0),
])
def test_ppo_backward_matches_fp64_autograd(n, noise, options, w_h):
    from wab_gym_b200.policy import PolicyTrainTC
    T = 24
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, options=options, head_scale=1.0)   # r can pass 1 + eps
    adv, target = _targets(T, n, seed=5)
    x = _materialise(env, feats, ctrs, noise)
    new, r = _perturbed(pol, x, acts, lp, adv)
    tc_new = PolicyTrainTC(env, new)
    # rows near a kink or within rounding of r = 1 +- eps are left out of the list (so out of both sides); the rest are
    # shuffled, half of them listed, with entries outside [0, T N) inside the count and padding beyond it
    bad = _near_kinks(new, x) | ((r - (1 + EPS)).abs() < 1e-3) | ((r - (1 - EPS)).abs() < 1e-3)
    assert float(bad.float().mean()) < 0.2
    g = torch.Generator(device="cuda").manual_seed(7)
    keep = torch.nonzero(~bad).squeeze(1)
    keep = keep[torch.randperm(keep.numel(), generator=g, device="cuda")][:keep.numel() // 2]
    sel = keep.sort().values
    a = adv.reshape(-1)[sel]
    assert float(((a > 0) & (r[sel] > 1 + EPS)).float().mean()) > 0.03 and float(((a < 0) & (r[sel] < 1 - EPS)).float().mean()) > 0.03
    outside = torch.tensor([-1, T * n, T * n + 5, -1000], dtype=torch.int32, device="cuda")
    listed = torch.cat([keep.to(torch.int32), outside])
    listed = listed[torch.randperm(listed.numel(), generator=g, device="cuda")]
    pad = torch.full((500,), 3, dtype=torch.int32, device="cuda")      # never read: beyond the count
    rows = torch.cat([listed, pad])
    n_rows = torch.tensor([listed.numel()], dtype=torch.int64, device="cuda")
    m = sel.numel()
    w = (1.0 / m, 0.5 / m, w_h / m)
    rlp, rv, ent = (torch.full_like(lp, float("nan")) for _ in range(3))
    grad = tc_new.ppo_backward(feats, ctrs, acts, lp, adv, target, rows, n_rows, EPS, *w, logp=rlp, value=rv, entropy=ent,
                               noise_scale=noise)
    assert torch.isfinite(grad).all()
    # V and log pi enter the upstream gradient, so the forward's own rounding does too: its truncating tensor-core
    # accumulation is a bias of ~1e-7 relative that a minibatch mean does not average out (torch's rounding does). The
    # references therefore evaluate the objective at the library forward's values (checked against fp64 below).
    _check_parity(new, grad, (x, acts, lp, adv, target, sel, w, (rlp, rv)))
    logq, v64, ent64 = _heads(copy.deepcopy(new).double(), x[sel].double())
    lp64 = logq.gather(1, acts.reshape(-1)[sel].long()[:, None]).squeeze(1)
    for got, want in ((rlp, lp64), (rv, v64), (ent, ent64)):
        assert torch.allclose(got.reshape(-1)[sel].double(), want, rtol=1e-5, atol=1e-5)
    unlisted = torch.ones(T * n, dtype=torch.bool, device="cuda")
    unlisted[sel] = False
    assert bool(torch.isnan(ent.reshape(-1)[unlisted]).all())   # only the listed rows are written
    env.close()


def test_ppo_backward_is_deterministic_and_a_zero_count_gives_zero():
    T, n = 16, 3000
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=4)
    adv, target = _targets(T, n, seed=6)
    rows = torch.randperm(T * n, device="cuda").to(torch.int32)
    cnt = torch.tensor([T * n // 2], dtype=torch.int64, device="cuda")
    args = (feats, ctrs, acts, lp - 0.1, adv, target, rows, cnt, EPS, 1e-3, 5e-4, 1e-5)
    a, b = tc.ppo_backward(*args), tc.ppo_backward(*args)
    assert torch.isfinite(a).all() and bool((a != 0).any()) and torch.equal(a, b)
    zero = tc.ppo_backward(*args[:7], torch.zeros(1, dtype=torch.int64, device="cuda"), *args[8:])
    assert torch.equal(zero, torch.zeros_like(zero))
    env.close()


def test_ppo_backward_stays_inside_its_buffers():
    T, n = 8, 1500
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=6)
    adv, target = _targets(T, n, seed=8)
    args = (feats, ctrs, acts, lp, adv, target, None, None, EPS, 1e-3, 5e-4, 1e-4)
    want_ent = torch.empty_like(lp)
    want = tc.ppo_backward(*args, entropy=want_ent)
    guard = 4096
    gbuf = torch.full((tc.n_params + 2 * guard,), 12345.0, device="cuda")
    ebuf = torch.full((T * n + 2 * guard,), -777.0, device="cuda")
    sbuf = torch.full((tc.scratch.numel() + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
    tc.scratch = sbuf[guard:guard + tc.scratch.numel()]
    got = tc.ppo_backward(*args, out=gbuf[guard:guard + tc.n_params], entropy=ebuf[guard:guard + T * n].view(T, n))
    torch.cuda.synchronize()
    assert torch.equal(got, want) and torch.equal(ebuf[guard:guard + T * n].view(T, n), want_ent)
    for buf, fill in ((gbuf, 12345.0), (ebuf, -777.0), (sbuf, 0xA5)):
        assert bool((buf[:guard] == fill).all()) and bool((buf[-guard:] == fill).all())
    env.close()


def test_ppo_backward_refuses_invalid_arguments():
    from wab_gym_b200.vec_env import _ptr
    T, n = 4, 512
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, 0.01, seed=9)
    adv, target = _targets(T, n, seed=10)
    grad = torch.empty(tc.n_params, device="cuda")
    w, b = tc.heads
    rows = torch.arange(T * n, dtype=torch.int32, device="cuda")
    cnt = torch.tensor([T * n], dtype=torch.int64, device="cuda")

    def call(**kw):
        a = dict(logp_old=_ptr(lp), adv=_ptr(adv), target=_ptr(target), rows=_ptr(rows), cnt=_ptr(cnt), eps=EPS, wp=1.0,
                 wv=0.5, wh=0.01, ent=None)
        a.update(kw)
        return tc.lib.wab_policy_ppo_backward(
            env._h, _ptr(feats), T, n, _ptr(ctrs), _ptr(acts), a["logp_old"], a["adv"], a["target"], a["rows"], a["cnt"],
            _ptr(tc.packed), _ptr(tc.bias), _ptr(tc.packed2), _ptr(tc.bias2), 150, _ptr(tc.packed3), _ptr(tc.bias3),
            _ptr(tc.packed2t), _ptr(tc.packed3t), _ptr(w), _ptr(b), w.shape[0] - 1, 0.01, 0.01, -4.0, 4.0, a["eps"], a["wp"],
            a["wv"], a["wh"], _ptr(tc.scratch), tc.scratch.numel(), _ptr(grad), None, None, a["ent"], None)

    assert call() == 0
    for k in ("logp_old", "adv", "target"):
        assert call(**{k: None}) == 1
    assert call(rows=None) == 1 and call(cnt=None) == 1           # rows and n_rows go together
    for k in ("logp_old", "adv", "target", "ent"):
        assert call(**{k: ctypes.c_void_p(lp.data_ptr() + 2)}) == 2
    for eps in (0.0, -0.1, float("nan"), float("-inf")):
        assert call(eps=eps) == 2
    assert call(eps=float("inf")) == 0
    for k in ("wp", "wv", "wh"):
        for bad in (float("inf"), float("-inf"), float("nan")):
            assert call(**{k: bad}) == 2
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        tc.ppo_backward(feats, ctrs, acts, lp, adv, target, rows, None, EPS, 1.0, 0.5, 0.0)
    with pytest.raises(ValueError):
        tc.ppo_backward(feats, ctrs, acts, lp.double(), adv, target, None, None, EPS, 1.0, 0.5, 0.0)
    with pytest.raises(ValueError):
        tc.ppo_backward(feats, ctrs, acts, lp, adv, target, None, None, 0.0, 1.0, 0.5, 0.0)
    env.close()


def _trainer(n, T, seed=2, **kw):
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    env = VecEnv(n, seed=seed, features=True, emit_grids=False)
    torch.manual_seed(seed)
    return PPOTrainer(env, Policy(env.flat_dim, env.n_actions).cuda(), horizon=T, **kw)


def test_trainer_gradient_matches_torch_replay():
    """epochs = minibatches = 1 without the norm clip: the trainer's gradient is that of ppo_loss replayed in torch on
    the recorded batch, GAE and normalisation included."""
    from wab_gym_b200.policy import PolicyTrainTC
    from wab_gym_b200.ppo import gae
    n, T = 2000, 32
    tr = _trainer(n, T, epochs=1, minibatches=1, max_grad_norm=float("inf"))
    before = copy.deepcopy(tr.policy)
    tr.env.stats(clear=True)
    info = tr.train_iteration()
    st = tr.env.stats()
    assert st["steps"] == n * T and st["bad_actions"] == 0
    assert float(info["clip_fraction"][0]) == 0.0 and float(info["approx_kl"][0]) == 0.0
    rec, env = tr.last_batch, tr.env
    x = _materialise(env, rec["features"], rec["counters"], 0.01)
    with torch.no_grad():
        logq, value, _ = _heads(before, x)
        boot = before(env.flatten_features_noisy(env.last_features, torch.empty(n, env.flat_dim, device="cuda"), 0.01, tr._ctr))[1]
    assert torch.allclose(logq.gather(1, rec["actions"].reshape(-1, 1).long()).squeeze(1), rec["logp"].reshape(-1), rtol=1e-5, atol=1e-5)
    assert torch.allclose(boot.squeeze(1), rec["bootstrap"], rtol=1e-5, atol=1e-5)
    adv, ret = gae(rec["reward"], rec["done"], rec["value"], rec["bootstrap"], tr.gamma, tr.lam)
    adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    assert torch.equal(adv, rec["advantage"]) and torch.equal(ret, rec["target"])
    # the trainer's gradient (p.grad, unscaled) against the library backward of the same batch over every row ...
    grad = torch.cat([p.grad.reshape(-1) for p in tr.policy.parameters()])
    m = T * n
    w = (1.0 / m, tr.vf_coef / m, tr.ent_coef / m)
    tc = PolicyTrainTC(env, before)
    full = tc.ppo_backward(rec["features"], rec["counters"], rec["actions"], rec["logp"], adv, ret, None, None, EPS, *w)
    assert torch.allclose(grad, full, rtol=1e-5, atol=1e-5 * float(full.abs().max()))
    # ... and that against fp64 autograd of ppo_loss on the off-kink rows
    sel = torch.nonzero(~_near_kinks(before, x)).squeeze(1)
    assert sel.numel() > 0.8 * m
    w = (1.0 / sel.numel(), tr.vf_coef / sel.numel(), tr.ent_coef / sel.numel())
    rows = sel.to(torch.int32)
    part = tc.ppo_backward(rec["features"], rec["counters"], rec["actions"], rec["logp"], adv, ret, rows,
                           torch.tensor([rows.numel()], dtype=torch.int64, device="cuda"), EPS, *w)
    _check_parity(before, part, (x, rec["actions"], rec["logp"], adv, ret, sel, w))
    env.close()


def test_trainer_runs_clips_and_resumes_bit_exactly():
    n, T, iters, kw = 1024, 16, 3, dict(epochs=2, minibatches=3)
    a = _trainer(n, T, **kw)
    p0 = [p.detach().clone() for p in a.policy.parameters()]
    a.env.stats(clear=True)
    for _ in range(iters):
        info = a.train_iteration()
        assert info["approx_kl"].shape == (6,) and float(info["clip_fraction"][0]) == 0.0 and float(info["approx_kl"][0]) == 0.0
        assert bool(torch.isfinite(info["policy_loss"]).all())
        norm = float(torch.linalg.vector_norm(torch.cat([p.grad.reshape(-1) for p in a.policy.parameters()])))
        assert norm <= a.max_grad_norm * (1 + 1e-5)
    st = a.env.stats()
    assert st["steps"] == n * T * iters and st["bad_actions"] == 0
    assert any(not torch.equal(p, q) for p, q in zip(p0, a.policy.parameters()))
    b = _trainer(n, T, **kw)
    for _ in range(2):
        b.train_iteration()
    sd = b.state_dict()
    b.env.close()
    c = _trainer(n, T, **kw)
    c.train_iteration()                                      # a state of its own first: everything comes from the state dict
    c.load_state_dict(sd)
    c.train_iteration()
    for p, q in zip(a.policy.parameters(), c.policy.parameters()):
        assert torch.equal(p, q)
    a.env.close(); c.env.close()


def test_trainer_refuses_what_the_kernels_do_not_cover():
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    env = VecEnv(256, seed=1, features=True)
    with pytest.raises(ValueError):
        PPOTrainer(env, Policy(env.flat_dim, env.n_actions).double())
    bad = Policy(env.flat_dim, env.n_actions)
    bad.affine2 = torch.nn.Linear(128, 140)
    with pytest.raises(ValueError):
        PPOTrainer(env, bad)
    with pytest.raises(ValueError):
        PPOTrainer(env, clip_eps=0.0)
    env.close()
    with pytest.raises(ValueError):
        PPOTrainer(VecEnv(256, seed=1))


def test_ppo_iteration_memory_is_within_one_and_a_half_of_a2c():
    from wab_gym_b200 import VecEnv
    from wab_gym_b200.a2c import A2CTrainer
    from wab_gym_b200.policy import Policy
    from wab_gym_b200.ppo import PPOTrainer
    peaks = {}
    for kind in ("a2c", "ppo"):
        env = VecEnv(32768, seed=3, features=True, emit_grids=False)
        torch.manual_seed(0)
        pol = Policy(env.flat_dim, env.n_actions)
        tr = A2CTrainer(env, pol, horizon=64, mode="horizon", tensor_cores=True) if kind == "a2c" else PPOTrainer(env, pol, horizon=64)
        tr.train_iteration()                                   # the first iteration allocates Adam's state
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        tr.train_iteration()
        torch.cuda.synchronize()
        peaks[kind] = torch.cuda.max_memory_allocated() - base
        env.close()
        del tr, env
        torch.cuda.empty_cache()
    print(peaks)
    assert peaks["ppo"] <= 1.5 * peaks["a2c"], peaks
