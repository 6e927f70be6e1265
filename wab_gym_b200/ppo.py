"""PPO on the tensor cores: several epochs of shuffled minibatches over one rollout, the clipped ratio objective, GAE
advantages and an entropy bonus (Schulman et al. 2017, "Proximal Policy Optimization Algorithms").

``PPOTrainer`` collects ``horizon`` steps of every environment with ``wab_policy_forward`` (one launch per step, keyed
sampling) and keeps what ``A2CTrainer(tensor_cores=True)`` keeps: 28 feature bytes, action, log-probability, value,
reward and done per env-step. Each minibatch is then ONE launch of ``wab_policy_ppo_backward``. It recomputes
log pi(a | x), V(x) and the entropy under the current weights and forms the clipped objective's upstream gradients in
the same registers, so no separate evaluation pass is needed for the ratio. The gradient is clipped by its global norm
on the device, and Adam steps on views of the flat gradient. Nothing in an iteration synchronises with the host.

``gae`` and ``ppo_loss`` are the torch statements of the advantage estimate and of the objective. ``ppo_loss`` is the
reference the tests differentiate, and the trainer's diagnostics.

Deliberate difference from CleanRL's ``ppo.py``: advantages are normalised once over the whole batch, not per
minibatch, so every minibatch of an iteration sees the same advantages. Value-loss clipping is not implemented.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch

from . import sharding
from .a2c import A2CTrainer
from .policy import Policy
from .vec_env import VecEnv


def gae(rewards: torch.Tensor, dones: torch.Tensor, values: torch.Tensor, bootstrap: torch.Tensor, gamma,
        lam: float, gamma_lam=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Generalised advantage estimation over [T, N] tensors: returns (advantages, returns = advantages + values).
    Step t's successor counts with the mask (1 - done_t): after a done the environment auto-resets, so nothing is
    bootstrapped across the boundary. A v1 episode that ends by ``max_turns`` is treated as terminal too. ``bootstrap``
    f32[N] is the value of the observation after the last step. Per-column discounts: ``gamma`` f32[N] and
    ``gamma_lam`` f32[N] (each column's gamma * lam, formed in double and rounded once, as a float gamma and lam are);
    ``lam`` is then unused."""
    T = rewards.shape[0]
    adv = torch.empty_like(rewards)
    running = torch.zeros_like(bootstrap)
    next_value = bootstrap
    gl = gamma * lam if gamma_lam is None else gamma_lam
    for t in range(T - 1, -1, -1):
        live = 1.0 - dones[t].to(rewards.dtype)
        delta = rewards[t] + gamma * next_value * live - values[t]
        running = delta + gl * live * running
        adv[t] = running
        next_value = values[t]
    return adv, adv + values


def ppo_loss(logp_new: torch.Tensor, value_new: torch.Tensor, entropy: torch.Tensor, logp_old: torch.Tensor,
             advantage: torch.Tensor, target: torch.Tensor, clip_eps: float, vf_coef: float,
             ent_coef: float) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """The mean over rows of  -min(r A, clip(r, 1 - eps, 1 + eps) A) + vf_coef (V - R)^2 / 2 - ent_coef H,
    r = exp(logp_new - logp_old). Returns (loss, diagnostics): policy and value loss, mean entropy, approx-KL
    mean((r - 1) - log r) and the fraction of rows with |r - 1| > eps."""
    log_ratio = logp_new - logp_old
    ratio = torch.exp(log_ratio)
    policy_loss = -torch.min(ratio * advantage, torch.clamp(ratio, 1.0 - clip_eps, 1.0 + clip_eps) * advantage).mean()
    value_loss = 0.5 * ((value_new - target) ** 2).mean()
    ent = entropy.mean()
    loss = policy_loss + vf_coef * value_loss - ent_coef * ent
    with torch.no_grad():
        info = {"policy_loss": policy_loss.detach(), "value_loss": value_loss.detach(), "entropy": ent.detach(),
                "approx_kl": ((ratio - 1.0) - log_ratio).mean(), "clip_fraction": ((ratio - 1.0).abs() > clip_eps).to(ratio.dtype).mean()}
    return loss, info


def _perm_seed(sample_seed: int, iteration: int, epoch: int, env_id_base=None) -> int:
    """The seed of an epoch's minibatch permutation. A rank of a data-parallel run (``env_id_base`` given) folds its
    first env id in, so that ranks shuffle differently; a single process keeps ``_seed(sample_seed, iteration, epoch)``."""
    return _seed(sample_seed, iteration, epoch) if env_id_base is None else _seed(sample_seed, iteration, epoch, env_id_base)


def _seed(*xs: int) -> int:
    """A 63-bit generator seed from integers (splitmix64 folded over them)."""
    h = 0x9E3779B97F4A7C15
    for x in xs:
        h = (h ^ (int(x) & 0xFFFFFFFFFFFFFFFF)) & 0xFFFFFFFFFFFFFFFF
        h = ((h ^ (h >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        h = ((h ^ (h >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        h ^= h >> 31
    return h & (2 ** 63 - 1)


class PPOTrainer(A2CTrainer):
    """PPO for N lockstep environments on this library's kernels; the reference's network only (it refuses what
    ``A2CTrainer(tensor_cores=True)`` refuses). Environments are never reset by the trainer: each iteration continues
    from where the last one stopped. Per iteration: collect ``horizon`` steps, GAE(gamma, lam) with the critic's value
    of the last observation as bootstrap, normalise the advantages over the batch, then ``epochs`` passes over a fresh
    permutation of the T N rows (``torch.Generator`` seeded by (sampling seed, iteration, epoch)), cut into
    ``minibatches`` contiguous slices. Each slice is one ``wab_policy_ppo_backward`` with the weights divided by its row
    count (the minibatch mean of ``ppo_loss``), a global-norm clip to ``max_grad_norm`` and an Adam step.

    With ``group`` (see ``a2c``'s module docstring) each rank runs GAE on its own envs, normalises the advantages by the
    mean and unbiased std of the whole batch, and permutes its own rows with ``env_id_base`` folded into the seed; every
    rank cuts its permutation into ``minibatches`` slices, and minibatch k's weights are divided by its row count summed
    over the ranks. After each ``wab_policy_ppo_backward`` the gradient is summed over the ranks (fp64, rank order, one
    rounding) before the clip and Adam, so the weights stay bit-identical on every rank. The returned diagnostics are
    this rank's rows, except ``grad_norm``, which is the global gradient's."""

    def __init__(self, env: VecEnv, policy: Policy = None, horizon: int = 64, epochs: int = 4, minibatches: int = 4,
                 gamma: float = 0.99, lam: float = 0.95, clip_eps: float = 0.2, vf_coef: float = 0.5, ent_coef: float = 0.01,
                 lr: float = 3e-4, max_grad_norm: float = 0.5, noise: bool = True, group=None):
        if epochs < 1 or minibatches < 1 or int(horizon) * env.num_envs < minibatches:
            raise ValueError("PPOTrainer needs epochs >= 1 and 1 <= minibatches <= horizon * num_envs")
        if not clip_eps > 0 or not max_grad_norm > 0:
            raise ValueError("clip_eps and max_grad_norm must be > 0")
        self.epochs, self.minibatches, self.lam = int(epochs), int(minibatches), float(lam)
        self.clip_eps, self.vf_coef, self.ent_coef, self.max_grad_norm = float(clip_eps), float(vf_coef), float(ent_coef), float(max_grad_norm)
        super().__init__(env, policy, horizon=horizon, gamma=gamma, lr=lr, noise=noise, mode="horizon", tensor_cores=True,
                         group=group)
        self.iteration = 0
        T, N, dev = self.horizon, env.num_envs, env.device
        rows = T * N
        self._bounds = sharding.minibatch_bounds(rows, self.minibatches)
        # the row count each minibatch's weights are divided by: this rank's, or the sum over the ranks (known from
        # construction, so no synchronisation)
        self._global_counts = ([self._bounds[k + 1] - self._bounds[k] for k in range(self.minibatches)] if self.group is None
                               else sharding.global_minibatch_counts([T * c for c in self._shard_counts], self.minibatches))
        self._counts = torch.tensor([self._bounds[k + 1] - self._bounds[k] for k in range(self.minibatches)], dtype=torch.int64, device=dev)
        self._new = {k: torch.empty(T, N, device=dev) for k in ("logp", "value", "entropy")}   # the kernel's per-row outputs
        self._perm = torch.empty(rows, dtype=torch.int32, device=dev)                          # this epoch's row order
        self.last_batch.update({"bootstrap": torch.empty(N, device=dev), "advantage": torch.empty(T, N, device=dev),
                                "target": torch.empty(T, N, device=dev)})
        self._rows = self._iota = None                   # A2C's row compaction is not used here
        off = 0
        for prm in self.policy.parameters():             # .grad = views of the flat gradient Adam steps on
            prm.grad = self._grad[off:off + prm.numel()].view_as(prm)
            off += prm.numel()

    def _signature(self) -> tuple:
        return super()._signature() + (self.epochs, self.minibatches, self.lam, self.clip_eps, self.vf_coef, self.ent_coef,
                                       self.max_grad_norm)

    def train_iteration(self) -> Dict[str, torch.Tensor]:
        """One PPO iteration. Returns device tensors: per minibatch (in order, ``epochs * minibatches`` entries) the
        ``ppo_loss`` diagnostics of its rows from the kernel's outputs and the gradient norm before clipping; the mean
        reward of the batch."""
        env, b, N = self.env, self.last_batch, self.env.num_envs
        noise = 0.01 if self.noise else 0.0
        self._collect_tc()
        self._sample_tc(env.last_features, self._boot_actions, b["bootstrap"])
        adv, ret = gae(b["reward"], b["done"], b["value"], b["bootstrap"], self.gamma, self.lam)
        b["target"].copy_(ret)
        if self.group is None:
            mean, std = adv.mean(), adv.std()
        else:
            mean, std = sharding.global_mean_std(adv, self.group)
        torch.sub(adv, mean, out=b["advantage"])                             # normalised once over the whole batch
        b["advantage"].div_(std + 1e-8)
        del adv, ret
        flat = {k: b[k].view(-1) for k in ("logp", "advantage", "target")}
        new = {k: v.view(-1) for k, v in self._new.items()}
        stats = []
        for epoch in range(self.epochs):
            gen = torch.Generator(device=env.device)
            gen.manual_seed(_perm_seed(self.sample_seed, self.iteration, epoch, None if self.group is None else env.env_id_base))
            torch.randperm(self._perm.numel(), generator=gen, out=self._perm)
            for k in range(self.minibatches):
                rows = self._perm[self._bounds[k]:self._bounds[k + 1]]
                m = float(self._global_counts[k])
                self._tc.ppo_backward(b["features"], b["counters"], b["actions"], b["logp"], b["advantage"], b["target"], rows,
                                      self._counts[k:k + 1], self.clip_eps, 1.0 / m, self.vf_coef / m, self.ent_coef / m,
                                      out=self._grad, logp=self._new["logp"], value=self._new["value"],
                                      entropy=self._new["entropy"], noise_scale=noise)
                if self.group is not None:
                    self._sum_grad_over_ranks()
                norm = torch.linalg.vector_norm(self._grad)
                self._grad.mul_(torch.clamp(self.max_grad_norm / (norm + 1e-6), max=1.0))
                self.optimizer.step()
                self._tc.refresh()
                _, info = ppo_loss(*(t.index_select(0, rows) for t in (new["logp"], new["value"], new["entropy"], flat["logp"],
                                                                      flat["advantage"], flat["target"])),
                                   self.clip_eps, self.vf_coef, self.ent_coef)
                info["grad_norm"] = norm
                stats.append(info)
        self.iteration += 1
        out = {k: torch.stack([s[k] for s in stats]) for k in stats[0]}
        out["mean_reward"] = b["reward"].mean()
        return out

    def state_dict(self) -> dict:
        """``A2CTrainer.state_dict`` (env, policy, Adam, noise counter, sampling seed) and the iteration counter that keys
        the minibatch permutations: a trainer resumed from it continues bit for bit."""
        sd = super().state_dict()
        sd["iteration"] = self.iteration
        return sd

    def load_state_dict(self, sd: dict):
        super().load_state_dict(sd)
        self.iteration = int(sd["iteration"])
