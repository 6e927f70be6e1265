"""PPO's advantage estimate and objective in torch (``wab_gym_b200.ppo``), on the CPU: GAE against a plain double loop,
``ppo_loss`` against hand-computed values, and autograd of ``ppo_loss`` against the closed-form per-row upstream
gradients that ``wab_policy_ppo_backward`` forms in its heads block."""
import math

import torch

from wab_gym_b200.ppo import gae, ppo_loss


def test_gae_equals_a_plain_double_loop():
    g = torch.Generator().manual_seed(0)
    T, N, gamma, lam = 9, 5, 0.97, 0.9
    rewards = torch.randn(T, N, generator=g)
    values = torch.randn(T, N, generator=g)
    bootstrap = torch.randn(N, generator=g)
    dones = torch.zeros(T, N, dtype=torch.bool)
    dones[2, 0] = dones[5, 0] = dones[T - 1, 1] = dones[0, 2] = dones[4, 3] = True      # mid-horizon, last step, first step
    adv, ret = gae(rewards, dones, values, bootstrap, gamma, lam)
    want = [[0.0] * N for _ in range(T)]
    for n in range(N):
        for t in range(T):
            a, discount = 0.0, 1.0
            for k in range(t, T):                                # sum_k (gamma lam)^(k - t) delta_k, stopped at a done
                nxt = float(bootstrap[n]) if k == T - 1 else float(values[k + 1, n])
                live = 0.0 if dones[k, n] else 1.0
                a += discount * (float(rewards[k, n]) + gamma * nxt * live - float(values[k, n]))
                if dones[k, n]:
                    break
                discount *= gamma * lam
            want[t][n] = a
    want = torch.tensor(want, dtype=torch.float64)
    assert torch.allclose(adv.double(), want, rtol=1e-5, atol=1e-5)
    assert torch.allclose(ret.double(), want + values.double(), rtol=1e-5, atol=1e-5)


def test_ppo_loss_by_hand():
    eps = 0.2
    r = torch.tensor([1.5, 0.5, 1.1, 1.5, 0.5, 1.0], dtype=torch.float64)
    adv = torch.tensor([2.0, -1.0, 1.0, -1.0, 2.0, -3.0], dtype=torch.float64)
    # clipped above (A > 0), clipped below (A < 0), unclipped, r above the band with A < 0, below with A > 0, r = 1
    per_row = [-(1.2 * 2.0), -(0.8 * -1.0), -1.1, -(1.5 * -1.0), -(0.5 * 2.0), -(1.0 * -3.0)]
    logp_old = torch.tensor([-0.3, -1.0, -2.0, -0.7, -0.1, -1.5], dtype=torch.float64)
    logp_new = logp_old + torch.log(r)
    value = torch.tensor([0.5, -1.0, 2.0, 0.0, 1.0, 3.0], dtype=torch.float64)
    target = torch.tensor([1.5, -1.0, 0.0, 0.5, 1.0, 1.0], dtype=torch.float64)
    ent = torch.tensor([1.0, 0.5, 1.5, 0.2, 0.1, 0.7], dtype=torch.float64)
    loss, info = ppo_loss(logp_new, value, ent, logp_old, adv, target, eps, 0.5, 0.01)
    pl = sum(per_row) / 6
    vl = 0.5 * (1.0 + 0.0 + 4.0 + 0.25 + 0.0 + 4.0) / 6
    el = float(ent.mean())
    assert math.isclose(float(info["policy_loss"]), pl, rel_tol=1e-12)
    assert math.isclose(float(info["value_loss"]), vl, rel_tol=1e-12)
    assert math.isclose(float(info["entropy"]), el, rel_tol=1e-12)
    assert math.isclose(float(loss), pl + 0.5 * vl - 0.01 * el, rel_tol=1e-12)
    kl = sum((x - 1.0) - math.log(x) for x in r.tolist()) / 6
    assert math.isclose(float(info["approx_kl"]), kl, rel_tol=1e-12)
    assert math.isclose(float(info["clip_fraction"]), 4 / 6, rel_tol=1e-12)     # |r - 1| > eps: 1.5, 0.5, 1.5, 0.5


def test_autograd_equals_the_closed_form_the_kernel_uses():
    """Per row with weights w_pi = 1/M, w_v = vf/M, w_H = ent/M (the minibatch mean):
    g_logp = -w_pi A r (0 where the clip is active), d logit_o = g_logp (1[o = a] - p_o) + w_H p_o (log p_o + H),
    d V = w_v (V - R)."""
    g = torch.Generator().manual_seed(1)
    M, A, eps, vf, ent_coef = 400, 6, 0.2, 0.5, 0.03
    logits = (2.0 * torch.randn(M, A, generator=g, dtype=torch.float64)).requires_grad_()
    logits.data[0, 0] = -800.0                                   # p underflows to 0: no NaN from 0 * log 0
    value = torch.randn(M, generator=g, dtype=torch.float64).requires_grad_()
    actions = torch.randint(0, A, (M,), generator=g)
    actions[0] = 1
    adv = torch.randn(M, generator=g, dtype=torch.float64)
    target = torch.randn(M, generator=g, dtype=torch.float64)
    logq = torch.log_softmax(logits, -1)
    logp_new = logq.gather(1, actions[:, None]).squeeze(1)
    logp_old = logp_new.detach() + 0.4 * torch.randn(M, generator=g, dtype=torch.float64)   # ratios on both sides of the band
    entropy = -(logq.exp() * logq).sum(-1)
    loss, _ = ppo_loss(logp_new, value, entropy, logp_old, adv, target, eps, vf, ent_coef)
    d_logits, d_value = torch.autograd.grad(loss, [logits, value])
    with torch.no_grad():
        w_pi, w_v, w_h = 1.0 / M, vf / M, ent_coef / M
        r = torch.exp(logp_new - logp_old)
        clipped = ((adv > 0) & (r > 1 + eps)) | ((adv < 0) & (r < 1 - eps))
        assert int(((adv > 0) & (r > 1 + eps)).sum()) > M // 20 and int(((adv < 0) & (r < 1 - eps)).sum()) > M // 20
        g_logp = torch.where(clipped, torch.zeros_like(r), -w_pi * adv * r)
        p = torch.softmax(logits, -1)
        log_p = (logits - logits.max(-1, keepdim=True).values) - torch.logsumexp(logits - logits.max(-1, keepdim=True).values, -1, keepdim=True)
        h = -(p * log_p).sum(-1, keepdim=True)
        onehot = torch.nn.functional.one_hot(actions, A).double()
        want_logits = g_logp[:, None] * (onehot - p) + w_h * p * (log_p + h)
        want_value = w_v * (value - target)
    assert torch.isfinite(d_logits).all()
    assert torch.allclose(d_logits, want_logits, rtol=1e-10, atol=1e-15)
    assert torch.allclose(d_value, want_value, rtol=1e-12, atol=1e-15)
