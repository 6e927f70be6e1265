"""Any loss through the tensor-core policy: ``PolicyTrainTC.logits_and_value`` (``wab_policy_evaluate`` forward,
``wab_policy_backward_logits`` backward) against the rollout, against fp64 autograd through ``Policy`` on the
materialised input, and against the fused A2C and PPO backward passes."""
import copy
import ctypes

import pytest
import torch
import torch.nn.functional as F

from tests.test_train_gpu import _materialise, _off_kinks, _record

pytestmark = pytest.mark.gpu

EPS = 0.2


def _keep(env, pol, feats, ctrs, noise):
    """_off_kinks' mask as bool[T N]: rows whose fp64 pre-activations are not within rounding of a kink."""
    T, n = feats.shape[:2]
    ones = torch.ones(T, n, device="cuda")
    keep, _, frac = _off_kinks(env, pol, feats, ctrs, ones, ones, noise)
    assert frac < 0.2, frac
    return keep.reshape(-1) != 0


def _outputs(p, x):
    """Policy.forward up to the heads: logits (before the softmax) and value."""
    h = F.leaky_relu(p.affine1(x))
    h = F.leaky_relu(p.affine2(h))
    h = torch.clamp(F.leaky_relu(p.affine3(h)), -4, 4)
    return p.action_head(h), p.value_head(h).squeeze(1)


def _ref_grads(pol, x, loss_fn, dtype, at=None):
    """Autograd of loss_fn(logits, value) through Policy in `dtype`. With `at` = (logits, value) of the library, the loss
    is evaluated at those values (the gradient still flows through Policy): an upstream that depends on the outputs then
    sees the same outputs on every side, and the comparison measures the backward pass alone."""
    p = copy.deepcopy(pol).to(dtype)
    logits, value = _outputs(p, x.to(dtype))
    if at is not None:
        logits = logits + (at[0].to(dtype) - logits).detach()
        value = value + (at[1].to(dtype) - value).detach()
    return torch.autograd.grad(loss_fn(logits, value), list(p.parameters()), allow_unused=True)


def _check_rule(pol, got, x, loss_fn, at=None, want=None):
    """test_train_gpu's parity rule per parameter tensor: |got - fp64| <= 2 |torch fp32 - fp64| + 1e-6 max |fp64|.
    With `want` given, the distance from `want` (another library gradient) is held to the same bound."""
    g64 = _ref_grads(pol, x, loss_fn, torch.float64, at)
    g32 = _ref_grads(pol, x, loss_fn, torch.float32, at)
    off, report, ok = 0, [], True
    for (name, prm), w64, w32 in zip(pol.named_parameters(), g64, g32):
        w64 = torch.zeros_like(prm, dtype=torch.float64) if w64 is None else w64
        w32 = torch.zeros_like(prm) if w32 is None else w32
        g = got[off:off + prm.numel()].view_as(prm).double()
        ref = w64 if want is None else want[off:off + prm.numel()].view_as(prm).double()
        off += prm.numel()
        err, err32, big = float((g - ref).abs().max()), float((w32.double() - w64).abs().max()), float(w64.abs().max())
        ok &= err <= 2 * err32 + 1e-6 * big
        report.append("%s: library error %.3g, torch fp32 error %.3g, largest %.3g" % (name, err, err32, big))
    assert off == got.numel()
    print("\n".join(report))
    assert ok, "\n".join(report)


def _flat_grad(pol):
    return torch.cat([p.grad.reshape(-1) for p in pol.parameters()])


def _lib_grad(tc, feats, ctrs, rows, loss_fn, noise=0.01):
    """The library's gradient of loss_fn through logits_and_value, and the outputs it was evaluated at."""
    for p in tc.policy.parameters():
        p.grad = None
    logits, value = tc.logits_and_value(feats, ctrs, rows, noise_scale=noise)
    loss_fn(logits, value).backward()
    return _flat_grad(tc.policy), (logits.detach(), value.detach())


@pytest.mark.parametrize("n,noise,options", [(1003, 0.01, None), (1000, 0.0, {"lookout_only": False}),
                                             (1000, 0.01, {"restrict_view": True})])
def test_evaluate_reproduces_the_rollout(n, noise, options):
    T = 16
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, options=options)
    with torch.no_grad():
        logits, value = tc.logits_and_value(feats, ctrs, noise_scale=noise)
    assert not logits.requires_grad and logits.shape == (T * n, env.n_actions) and value.shape == (T * n,)
    assert torch.equal(value, v.reshape(-1))                      # the rollout's forward, bit for bit
    logq = torch.log_softmax(logits, -1).gather(1, acts.reshape(-1, 1).long()).squeeze(1)
    assert float((logq - lp.reshape(-1)).abs().max()) <= 1e-6
    x = _materialise(env, feats, ctrs, noise).reshape(T * n, -1)
    with torch.no_grad():
        want, _ = _outputs(copy.deepcopy(pol).double(), x.double())
    assert float((logits.double() - want).abs().max()) <= 3e-6 * max(float(want.abs().max()), 1.0)
    # a shuffled, ragged list with repeats and entries outside [0, T N)
    g = torch.Generator(device="cuda").manual_seed(3)
    perm = torch.randperm(T * n, generator=g, device="cuda")[:T * n // 3]
    bad = torch.tensor([-1, T * n, T * n + 7, -100000], device="cuda")
    rows = torch.cat([perm, perm[:301], bad])
    rows = rows[torch.randperm(rows.numel(), generator=g, device="cuda")].to(torch.int32)
    assert rows.numel() % 128 != 0
    with torch.no_grad():
        lg, vl = tc.logits_and_value(feats, ctrs, rows, noise_scale=noise)
    inside = (rows >= 0) & (rows < T * n)
    r = rows[inside].long()
    assert torch.equal(lg[inside], logits[r]) and torch.equal(vl[inside], value[r])
    assert bool(torch.isnan(lg[~inside]).all()) and bool(torch.isnan(vl[~inside]).all()) and int((~inside).sum()) == 4
    env.close()


@pytest.mark.parametrize("n,noise,options", [(1000, 0.0, None), (1003, 0.01, None), (1000, 0.01, {"lookout_only": False}),
                                             (1000, 0.01, {"restrict_view": True})])
def test_vector_jacobian_product_matches_fp64_autograd(n, noise, options):
    T = 24
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, options=options)
    sel = torch.nonzero(_keep(env, pol, feats, ctrs, noise)).squeeze(1)
    x = _materialise(env, feats, ctrs, noise).reshape(T * n, -1)[sel]
    g = torch.Generator(device="cuda").manual_seed(5)
    g_logits = torch.randn(sel.numel(), env.n_actions, device="cuda", generator=g)
    g_value = torch.randn(sel.numel(), device="cuda", generator=g)

    def loss_fn(logits, value):
        return (logits * g_logits.to(logits.dtype)).sum() + (value * g_value.to(value.dtype)).sum()

    got, _ = _lib_grad(tc, feats, ctrs, sel.to(torch.int32), loss_fn, noise)
    assert torch.isfinite(got).all()
    _check_rule(pol, got, x, loss_fn)
    env.close()


def _perturbed(pol, seed=11, c=0.3):
    """A copy of `pol` moved so that ratios and values spread from the recorded ones."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    p = copy.deepcopy(pol)
    with torch.no_grad():
        for prm in p.parameters():
            prm.add_(1e-3 * prm.abs().mean() * torch.randn(prm.shape, device="cuda", generator=g))
        p.action_head.weight.add_(c * torch.randn(p.action_head.weight.shape, device="cuda", generator=g))
        p.value_head.weight.add_(c * torch.randn(p.value_head.weight.shape, device="cuda", generator=g))
    return p


def _ppo_value_clip_loss(logp_old, v_old, adv, target, acts, ent_coef=0.01, vf_coef=0.5):
    """CleanRL's PPO: advantages normalised per minibatch, the clipped value loss, an entropy bonus."""
    def loss_fn(logits, value):
        dt = logits.dtype
        logq = torch.log_softmax(logits, -1)
        logp = logq.gather(1, acts[:, None]).squeeze(1)
        a = adv.to(dt)
        a = (a - a.mean()) / (a.std() + 1e-8)
        ratio = torch.exp(logp - logp_old.to(dt))
        pg = torch.max(-a * ratio, -a * torch.clamp(ratio, 1 - EPS, 1 + EPS)).mean()
        vo, R = v_old.to(dt), target.to(dt)
        v_clip = vo + torch.clamp(value - vo, -EPS, EPS)
        vl = 0.5 * torch.max((value - R) ** 2, (v_clip - R) ** 2).mean()
        ent = -(logq.exp() * logq).sum(-1).mean()
        return pg + vf_coef * vl - ent_coef * ent
    return loss_fn


@pytest.mark.parametrize("loss", ["ppo_value_clip_entropy", "cross_entropy_kl", "value_smooth_l1"])
def test_losses_users_write_match_fp64_autograd(loss):
    from wab_gym_b200.policy import PolicyTrainTC
    T, n, noise = 16, 1500, 0.01
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, seed=2)
    new = _perturbed(pol)
    tc_new = PolicyTrainTC(env, new)
    sel = torch.nonzero(_keep(env, new, feats, ctrs, noise)).squeeze(1)
    g = torch.Generator(device="cuda").manual_seed(7)
    sel = sel[torch.randperm(sel.numel(), generator=g, device="cuda")][:sel.numel() // 2]
    x = _materialise(env, feats, ctrs, noise).reshape(T * n, -1)[sel]
    m, A = sel.numel(), env.n_actions
    a = acts.reshape(-1)[sel].long()
    if loss == "ppo_value_clip_entropy":
        adv = torch.randn(m, device="cuda", generator=g) + 0.3
        target = v.reshape(-1)[sel] + torch.randn(m, device="cuda", generator=g)
        loss_fn = _ppo_value_clip_loss(lp.reshape(-1)[sel], v.reshape(-1)[sel], adv, target, a)
    elif loss == "cross_entropy_kl":
        tgt = torch.randint(0, A, (m,), device="cuda", generator=g)
        q = torch.softmax(torch.randn(m, A, device="cuda", generator=g), -1)

        def loss_fn(logits, value):
            logq = torch.log_softmax(logits, -1)
            kl = (q.to(logits.dtype) * (torch.log(q.to(logits.dtype)) - logq)).sum(-1).mean()
            return F.cross_entropy(logits, tgt) + 0.1 * kl
    else:
        target = v.reshape(-1)[sel] + 2.0 * torch.randn(m, device="cuda", generator=g)

        def loss_fn(logits, value):
            return F.smooth_l1_loss(value, target.to(value.dtype))
    got, at = _lib_grad(tc_new, feats, ctrs, sel.to(torch.int32), loss_fn, noise)
    assert torch.isfinite(got).all() and bool((got != 0).any())
    if loss == "ppo_value_clip_entropy":                          # both clips active on some rows
        logp = torch.log_softmax(at[0], -1).gather(1, a[:, None]).squeeze(1)
        r = torch.exp(logp - lp.reshape(-1)[sel])
        assert float(((r - 1).abs() > EPS).float().mean()) > 0.03
        assert float(((at[1] - v.reshape(-1)[sel]).abs() > EPS).float().mean()) > 0.03
    _check_rule(new, got, x, loss_fn, at=at)
    if loss == "value_smooth_l1":                                 # no upstream into the logits: exactly zero
        off = sum(p.numel() for p in list(new.parameters())[:6])
        n_ah = A * 128 + A
        assert bool((got[off:off + n_ah] == 0).all()) and bool((got[off + n_ah:] != 0).any())
    env.close()


def test_agrees_with_the_fused_a2c_backward():
    T, n, noise = 24, 1500, 0.01
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, seed=4)
    g = torch.Generator(device="cuda").manual_seed(9)
    gl, gv, _ = _off_kinks(env, pol, feats, ctrs, torch.randn(T, n, device="cuda", generator=g),
                           torch.randn(T, n, device="cuda", generator=g), noise)
    a = acts.reshape(-1).long()

    def loss_fn(logits, value):
        logp = torch.log_softmax(logits, -1).gather(1, a[:, None]).squeeze(1)
        return (gl.reshape(-1).to(logits.dtype) * logp).sum() + (gv.reshape(-1).to(value.dtype) * value).sum()

    got, at = _lib_grad(tc, feats, ctrs, None, loss_fn, noise)
    fused = tc.backward(feats, ctrs, acts, gl, gv, noise_scale=noise)
    x = _materialise(env, feats, ctrs, noise).reshape(T * n, -1)
    _check_rule(pol, got, x, loss_fn, at=at, want=fused)
    env.close()


def test_agrees_with_the_fused_ppo_backward():
    from wab_gym_b200.policy import PolicyTrainTC
    from wab_gym_b200.ppo import ppo_loss
    T, n, noise = 16, 2000, 0.01
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, seed=6)
    new = _perturbed(pol, seed=12, c=0.1)
    tc_new = PolicyTrainTC(env, new)
    g = torch.Generator(device="cuda").manual_seed(13)
    adv, target = torch.randn(T, n, device="cuda", generator=g), torch.randn(T, n, device="cuda", generator=g)
    # rows near a kink or within rounding of r = 1 +- eps (where the two sides may clip differently) are left out
    with torch.no_grad():
        lg, _ = tc_new.logits_and_value(feats, ctrs, noise_scale=noise)
    r = torch.exp(torch.log_softmax(lg, -1).gather(1, acts.reshape(-1, 1).long()).squeeze(1) - lp.reshape(-1))
    near_clip = ((r - (1 + EPS)).abs() < 1e-3) | ((r - (1 - EPS)).abs() < 1e-3)
    sel = torch.nonzero(_keep(env, new, feats, ctrs, noise) & ~near_clip).squeeze(1)
    sel = sel[torch.randperm(sel.numel(), generator=g, device="cuda")][:sel.numel() // 4]
    rows, m = sel.to(torch.int32), sel.numel()
    a = acts.reshape(-1)[sel].long()
    vf, ent_c = 0.5, 0.01

    def loss_fn(logits, value):
        logq = torch.log_softmax(logits, -1)
        ent = -(logq.exp() * logq).sum(-1)
        dt = logits.dtype
        loss, _ = ppo_loss(logq.gather(1, a[:, None]).squeeze(1), value, ent, lp.reshape(-1)[sel].to(dt),
                           adv.reshape(-1)[sel].to(dt), target.reshape(-1)[sel].to(dt), EPS, vf, ent_c)
        return loss

    got, at = _lib_grad(tc_new, feats, ctrs, rows, loss_fn, noise)
    fused = tc_new.ppo_backward(feats, ctrs, acts, lp, adv, target, rows, torch.tensor([m], dtype=torch.int64, device="cuda"),
                                EPS, 1.0 / m, vf / m, ent_c / m, noise_scale=noise)
    x = _materialise(env, feats, ctrs, noise).reshape(T * n, -1)[sel]
    _check_rule(new, got, x, loss_fn, at=at, want=fused)
    env.close()


def test_autograd_semantics():
    from wab_gym_b200.policy import PolicyTrainTC
    T, n, noise = 8, 1200, 0.01
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, seed=8)
    rows = torch.randperm(T * n, device="cuda")[:5000].to(torch.int32)
    w = torch.randn(5000, env.n_actions, device="cuda")

    def loss_of(t):
        logits, value = t.logits_and_value(feats, ctrs, rows, noise_scale=noise)
        return (logits * w).sum() + value.square().sum()

    # two backward passes accumulate exactly twice one pass
    loss_of(tc).backward()
    one = [p.grad.clone() for p in pol.parameters()]
    loss_of(tc).backward()
    for p, g1 in zip(pol.parameters(), one):
        assert torch.equal(p.grad, 2 * g1)
    # torch.autograd.grad for a subset of the parameters
    sub = torch.autograd.grad(loss_of(tc), [pol.affine2.weight, pol.value_head.bias])
    assert torch.equal(sub[0], one[2]) and torch.equal(sub[1], one[9])
    # after an optimiser step the next call uses the new weights, with no refresh()
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3)
    opt.step()
    for p in pol.parameters():
        p.grad = None
    loss_of(tc).backward()
    after = [p.grad.clone() for p in pol.parameters()]
    fresh_pol = copy.deepcopy(pol)
    fresh = PolicyTrainTC(env, fresh_pol)
    loss_of(fresh).backward()
    for p, q in zip(after, fresh_pol.parameters()):
        assert torch.equal(p, q.grad)
    with torch.no_grad():
        assert all(torch.equal(s, f) for s, f in zip(tc.logits_and_value(feats, ctrs, rows, noise_scale=noise),
                                                     fresh.logits_and_value(feats, ctrs, rows, noise_scale=noise)))
    # an in-place change between the forward and the backward raises autograd's version error
    loss = loss_of(tc)
    with torch.no_grad():
        pol.affine1.bias.add_(1.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        loss.backward()
    # nothing synchronises with the host
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        logits, value = tc.logits_and_value(feats, ctrs, rows, noise_scale=noise)
        torch.autograd.backward([logits, value], [w, torch.ones_like(value)])
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    env.close()


def test_repeated_calls_are_bit_identical_and_grad_f64_sums_to_the_same():
    T, n, noise = 8, 2100, 0.01
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, seed=10)
    rows = torch.randperm(T * n, device="cuda")[:9999].to(torch.int32)
    w = torch.randn(9999, env.n_actions, device="cuda")
    runs = []
    for _ in range(3):
        for p in pol.parameters():
            p.grad = None
        logits, value = tc.logits_and_value(feats, ctrs, rows, noise_scale=noise)
        ((logits * w).sum() + (value * value).sum()).backward()
        runs.append((logits.detach(), value.detach(), _flat_grad(pol)))
    for r in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(runs[0], r))
    # the scratch of the last logits backward reduces in fp64 to the same gradient, rounded once (one rank)
    g64 = tc.grad_f64()
    assert torch.equal(tc.grad_sum_ranks(g64[None].contiguous()), runs[0][2]) and torch.equal(g64.float(), runs[0][2])
    env.close()


def _abi(tc, env, features, counters, T, n, **kw):
    """Both entry points through the C ABI with every argument overridable."""
    from wab_gym_b200.vec_env import _ptr
    w, b = tc.heads
    a = dict(h=env._h, feats=_ptr(features), T=T, n=n, ctrs=_ptr(counters), rows=None, m=T * n, gl=None, gv=None,
             p1=_ptr(tc.packed), p2=_ptr(tc.packed2), p3=_ptr(tc.packed3), p2t=_ptr(tc.packed2t), p3t=_ptr(tc.packed3t),
             hidden2=150, A=w.shape[0] - 1, noise=0.01, scratch=_ptr(tc.scratch), sbytes=tc.scratch.numel(),
             logits=None, value=None, grad=None)
    a.update(kw)
    if a["logits"] is not None:
        return tc.lib.wab_policy_evaluate(
            a["h"], a["feats"], a["T"], a["n"], a["ctrs"], a["rows"], a["m"], a["p1"], _ptr(tc.bias), a["p2"], _ptr(tc.bias2),
            a["hidden2"], a["p3"], _ptr(tc.bias3), _ptr(w), _ptr(b), a["A"], a["noise"], 0.01, -4.0, 4.0, a["scratch"],
            a["sbytes"], a["logits"], a["value"], None)
    return tc.lib.wab_policy_backward_logits(
        a["h"], a["feats"], a["T"], a["n"], a["ctrs"], a["rows"], a["m"], a["gl"], a["gv"], a["p1"], _ptr(tc.bias), a["p2"],
        _ptr(tc.bias2), a["hidden2"], a["p3"], _ptr(tc.bias3), a["p2t"], a["p3t"], _ptr(w), _ptr(b), a["A"], a["noise"], 0.01,
        -4.0, 4.0, a["scratch"], a["sbytes"], a["grad"], None)


def test_stays_inside_its_buffers_and_refuses_invalid_arguments():
    from wab_gym_b200.vec_env import _ptr
    T, n, noise = 6, 1500, 0.01
    env, pol, tc, feats, ctrs, acts, lp, v = _record(n, T, noise, seed=12)
    M, A, guard = T * n, env.n_actions, 4096
    g_logits = torch.randn(M, A, device="cuda")
    g_value = torch.randn(M, device="cuda")
    with torch.no_grad():
        want_l, want_v = tc.logits_and_value(feats, ctrs, noise_scale=noise)
    want_g = torch.empty(tc.n_params, device="cuda")
    assert _abi(tc, env, feats, ctrs, T, n, gl=_ptr(g_logits), gv=_ptr(g_value), grad=_ptr(want_g)) == 0
    lbuf = torch.full((M * A + 2 * guard,), -777.0, device="cuda")
    vbuf = torch.full((M + 2 * guard,), -777.0, device="cuda")
    gbuf = torch.full((tc.n_params + 2 * guard,), 12345.0, device="cuda")
    sbuf = torch.full((tc.scratch.numel() + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
    tc.scratch = sbuf[guard:guard + tc.scratch.numel()]
    assert _abi(tc, env, feats, ctrs, T, n, logits=_ptr(lbuf[guard:]), value=_ptr(vbuf[guard:])) == 0
    assert _abi(tc, env, feats, ctrs, T, n, gl=_ptr(g_logits), gv=_ptr(g_value), grad=_ptr(gbuf[guard:])) == 0
    torch.cuda.synchronize()
    assert torch.equal(lbuf[guard:guard + M * A].view(M, A), want_l) and torch.equal(vbuf[guard:guard + M], want_v)
    assert torch.equal(gbuf[guard:guard + tc.n_params], want_g)
    for buf, fill in ((lbuf, -777.0), (vbuf, -777.0), (gbuf, 12345.0), (sbuf, 0xA5)):
        assert bool((buf[:guard] == fill).all()) and bool((buf[-guard:] == fill).all())
    # refusals: 1 WAB_E_NULL, 2 WAB_E_CONFIG, 3 WAB_E_UNSUPPORTED
    lo, va, gr = torch.empty(M, A, device="cuda"), torch.empty(M, device="cuda"), torch.empty(tc.n_params, device="cuda")
    ev = dict(logits=_ptr(lo), value=_ptr(va))
    bw = dict(gl=_ptr(g_logits), gv=_ptr(g_value), grad=_ptr(gr))
    odd = ctypes.c_void_p(lo.data_ptr() + 2)
    for kw in (ev, bw):
        assert _abi(tc, env, feats, ctrs, T, n, **kw) == 0
        for k in ("h", "feats", "ctrs", "p1", "p2", "p3", "scratch"):
            assert _abi(tc, env, feats, ctrs, T, n, **{**kw, k: None}) == 1, k
        assert _abi(tc, env, feats, ctrs, T, n, **{**kw, "m": -1}) == 2
        for bad in (-0.01, float("nan"), float("inf")):
            assert _abi(tc, env, feats, ctrs, T, n, **{**kw, "noise": bad}) == 2
        assert _abi(tc, env, feats, ctrs, T, n, **{**kw, "sbytes": tc.scratch.numel() - 1}) == 2
        assert _abi(tc, env, feats, ctrs, T, n, **{**kw, "scratch": ctypes.c_void_p(tc.scratch.data_ptr() + 4)}) == 2
        assert _abi(tc, env, feats, ctrs, T, n, **{**kw, "rows": odd}) == 2
        assert _abi(tc, env, feats, ctrs, T, n, **{**kw, "A": 9}) == 3
        assert _abi(tc, env, feats, ctrs, T, n, **{**kw, "hidden2": 140}) == 3
    assert _abi(tc, env, feats, ctrs, T, n, logits=_ptr(lo), value=None) == 1
    assert _abi(tc, env, feats, ctrs, T, n, logits=odd, value=_ptr(va)) == 2
    for k in ("gl", "gv", "grad", "p2t", "p3t"):
        assert _abi(tc, env, feats, ctrs, T, n, **{**bw, k: None}) == 1, k
    for k in ("gl", "gv", "grad"):
        assert _abi(tc, env, feats, ctrs, T, n, **{**bw, k: odd}) == 2, k
    torch.cuda.synchronize()
    # the Python layer validates shapes and dtypes
    for args in ((feats[..., :27], ctrs), (feats, ctrs.int()), (feats, ctrs[:-1]), (feats.float(), ctrs)):
        with pytest.raises(ValueError):
            tc.logits_and_value(*args)
    with pytest.raises(ValueError):
        tc.logits_and_value(feats, ctrs, torch.arange(10, device="cuda"))
    with pytest.raises(ValueError):
        tc.logits_and_value(feats, ctrs, noise_scale=-1.0)
    env.close()
