"""Batched on-device actor-critic update — the reference's ``finish_episode`` (``actor_critic.py:128-169``)
for N lockstep environments.

The reference trains on ONE environment, one episode per update: discounted Monte-Carlo returns over the episode
(``:139-144``), normalised by the episode's own mean and (unbiased) standard deviation (``:146-147``), policy loss
``-log_prob * (R - value.item())`` (``:150-153``), critic loss ``smooth_l1(value, R)`` (``:156``), both SUMMED over
the episode (``:162``), Adam (``:159-165``); it synchronises with the host at every step (``.item()``, ``:125``) and
walks Python lists per episode (``:139-155``).

``episodic_actor_critic_loss`` is that loss for a batch of episodes at once — the sum over episodes of the
reference's per-episode loss (N episodes accumulated into one optimiser step; with N = 1 it IS ``finish_episode``).
``A2CTrainer.train_iteration`` collects one episode per environment with every tensor on the device: all
environments are reset together, stepped ``max_turns`` times (every v1 episode ends by then, ``wab_env.py:328-340``)
and each environment contributes the steps up to and including its first ``done``; what an auto-reset environment
does after that is masked out. The policy input is the keyed flatten + noise kernel of the rollout
(``actor_critic.py:188-189``). Deliberate difference: an episode of length 1 has no standard deviation (the
reference computes ``nan`` there and poisons its weights); such episodes are left out of the loss and counted.

``mode="horizon"`` keeps the fixed-horizon variant of round 1 (returns restart at episode boundaries, the unfinished
tail is bootstrapped with the critic) — a different estimator, not the reference's update.

``tensor_cores=True`` trains on this library's kernels: collection is ``wab_policy_forward`` (one tcgen05 launch per step,
keyed sampling), the loss is the same torch code on the recorded log-probabilities and values as leaves, and the backward
pass is ``wab_policy_backward``, which recomputes the forward from the 28 feature bytes of every step instead of keeping
autograd's activations (62 bytes per env-step instead of about 5.5 KB). It serves the reference's network only.

Data-parallel training (``group``, a ``torch.distributed`` process group; ``tensor_cores=True`` only): each rank holds one
contiguous shard of global env ids, ``VecEnv(count, env_id_base=first)`` with ``sharding.shard_range``. Construction
checks on every rank that the shards tile ``[0, total)`` in rank order and that the trainers agree (options fingerprint,
horizon, hyper-parameters, action count), then broadcasts rank 0's weights and sampling seed. The policy's draws are
keyed by the global env id, so collection is invariant to the world size: rank r records exactly rows
``[first_r, first_r + count_r)`` of a single-process run with the same weights. Every cross-rank sum (the gradient, the
normalisation statistics of horizon mode and of PPO) is an all-gather followed by a sum in rank order in fp64 on every
rank, so every rank holds bit-identical weights after every step. Training is deterministic for a fixed shard layout and
resumes bit for bit on it; it is NOT bit-exact across world sizes (the tensor-core weight gradient rounds per 128-row
tile in fp32, and the tiles hold other rows under another layout; PPO's minibatches depend on the layout). A checkpoint
merged with ``sharding.merge_trainer_state_dicts`` resumes on any layout, a single process included, and its next
collected batch equals the uninterrupted run's. Returned diagnostics describe this rank's rows, except ``grad_norm``
(PPO), which is global.
"""
from __future__ import annotations

import copy
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

from . import sharding
from .policy import Policy, PolicyTrainTC, check_reference_network
from .vec_env import VecEnv


def episodic_actor_critic_loss(log_probs: torch.Tensor, values: torch.Tensor, rewards: torch.Tensor, dones: torch.Tensor,
                               gamma: float, eps: float) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """``finish_episode`` (``actor_critic.py:128-165``) for N episodes laid out as [T, N] tensors: env n's episode is
    steps 0 .. first done (inclusive); later steps are ignored. Returns (loss, diagnostics)."""
    T, N = rewards.shape
    d = dones.to(torch.bool)
    ended_before = torch.cumsum(d.to(torch.int32), 0) - d.to(torch.int32)      # dones strictly before step t
    mask = ended_before == 0                                                   # steps of the first episode
    complete = d.any(0)                                                        # envs whose episode ended inside T
    mask = mask & complete
    m = mask.to(rewards.dtype)
    returns = torch.zeros_like(rewards)
    running = torch.zeros(N, dtype=rewards.dtype, device=rewards.device)
    for t in range(T - 1, -1, -1):                                             # R = r + gamma * R  (:139-144)
        running = (rewards[t] + gamma * running) * m[t]
        returns[t] = running
    length = m.sum(0)
    usable = length >= 2                                                       # std of one sample is nan (:147)
    m = m * usable.to(m.dtype)
    safe_len = length.clamp(min=2)
    mean = (returns * m).sum(0) / safe_len
    var = (((returns - mean) * m) ** 2).sum(0) / (safe_len - 1)                # torch.std: unbiased
    norm = (returns - mean) / (var.sqrt() + eps)                               # :146-147
    advantage = norm - values.detach()                                         # R - value.item(), :150
    policy_loss = (-(log_probs * advantage) * m).sum()                         # :153, :162
    value_loss = (F.smooth_l1_loss(values, norm, reduction="none") * m).sum()  # :156, :162
    return policy_loss + value_loss, {"policy_loss": policy_loss.detach(), "value_loss": value_loss.detach(),
                                      "episodes": usable.sum(), "skipped_single_step": (complete & ~usable).sum(),
                                      "mean_length": (length * usable).sum() / usable.sum().clamp(min=1)}


def horizon_returns(rewards: torch.Tensor, dones: torch.Tensor, bootstrap: torch.Tensor, gamma: float) -> torch.Tensor:
    """Discounted returns over [T, N] tensors, restarted at done, the tail bootstrapped with ``bootstrap`` f32[N]."""
    T, N = rewards.shape
    with torch.no_grad():
        running = bootstrap
        returns = torch.empty(T, N, device=rewards.device)
        for t in range(T - 1, -1, -1):                                       # R = r + gamma * R, restarted at done
            running = rewards[t] + gamma * running * (~dones[t]).float()
            returns[t] = running
    return returns


def horizon_actor_critic_loss(log_probs: torch.Tensor, values: torch.Tensor, rewards: torch.Tensor, dones: torch.Tensor,
                              bootstrap: torch.Tensor, gamma: float, eps: float, mean: Optional[torch.Tensor] = None,
                              std: Optional[torch.Tensor] = None,
                              total_envs: Optional[int] = None) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """The fixed-horizon loss of ``mode="horizon"``: returns restart at done, the tail is bootstrapped with ``bootstrap``.
    The returns are normalised by their mean and unbiased std over this batch, or by ``mean`` / ``std`` when given (those
    of a data-parallel run's whole batch); the mean over environments divides by ``total_envs`` when given (the run's
    environment count, so that the ranks' losses add up to the whole batch's)."""
    returns = horizon_returns(rewards, dones, bootstrap, gamma)
    with torch.no_grad():
        if mean is None:
            returns = (returns - returns.mean()) / (returns.std() + eps)
        else:
            returns = (returns - mean) / (std + eps)
    advantage = returns - values.detach()
    if total_envs is None:
        policy_loss = -(log_probs * advantage).sum(0).mean()
        value_loss = F.smooth_l1_loss(values, returns, reduction="none").sum(0).mean()
    else:
        policy_loss = -(log_probs * advantage).sum() / total_envs
        value_loss = F.smooth_l1_loss(values, returns, reduction="none").sum() / total_envs
    return policy_loss + value_loss, {"policy_loss": policy_loss.detach(), "value_loss": value_loss.detach()}


class A2CTrainer:
    def __init__(self, env: VecEnv, policy: Policy = None, horizon: int = None, gamma: float = 0.99, lr: float = 3e-2,
                 noise: bool = True, mode: str = "episodic", tensor_cores: bool = False, group=None):
        if not env.with_features:
            raise ValueError("A2CTrainer needs VecEnv(features=True)")
        if getattr(env, "replicas", 1) > 1:
            raise ValueError("the trainers refuse a VecEnv with replicas: its env ids repeat")
        if mode not in ("episodic", "horizon"):
            raise ValueError("mode must be 'episodic' or 'horizon'")
        self.env, self.gamma, self.noise, self.mode = env, float(gamma), noise, mode
        self.horizon = int(horizon) if horizon is not None else int(env.game_options["max_turns"])
        self.policy = (policy or Policy(env.flat_dim, env.n_actions)).to(env.device)
        self.optimizer = torch.optim.Adam(self.policy.parameters(), lr=lr)      # actor_critic.py:103 (lr = 3e-2)
        self.eps = torch.finfo(torch.float32).eps                                # :104
        self._flat = torch.empty(env.num_envs, env.flat_dim, dtype=torch.float32, device=env.device)
        self._ctr = torch.zeros(1, dtype=torch.int64, device=env.device)
        self.tensor_cores = bool(tensor_cores)
        self.sample_seed = int(torch.initial_seed()) & (2 ** 63 - 1)
        self.group = group if sharding._distributed(group) else None
        if self.group is not None and not self.tensor_cores:
            raise ValueError("data-parallel training (a group of more than one rank) needs tensor_cores=True")
        if self.tensor_cores:
            self._init_tensor_cores()
        env.reset()
        if self.group is not None:
            self._join_group()

    def _signature(self) -> tuple:
        """What every rank of a data-parallel run must agree on."""
        return (self.env.fingerprint, self.env.n_actions, self.horizon, self.mode, self.gamma, bool(self.noise),
                float(self.optimizer.param_groups[0]["lr"]))

    def _join_group(self):
        """Validate the shard layout and the trainers on every rank (one host synchronisation), then take rank 0's
        weights and sampling seed."""
        import torch.distributed as dist
        world, env = dist.get_world_size(self.group), self.env
        infos = [None] * world
        dist.all_gather_object(infos, (env.env_id_base, env.num_envs, self._signature()), group=self.group)
        self.total_envs = sharding.check_trainer_shards(infos)
        self._shard_counts = [int(c) for _, c, _ in infos]
        src = dist.get_global_rank(self.group, 0)
        with torch.no_grad():
            for prm in self.policy.parameters():
                dist.broadcast(prm.data, src, group=self.group)
        seed = torch.tensor([self.sample_seed], dtype=torch.int64, device=env.device)
        dist.broadcast(seed, src, group=self.group)
        self.sample_seed = int(seed.item())
        self._tc.refresh()
        self._grad64 = torch.empty(self._tc.n_params, dtype=torch.float64, device=env.device)
        self._gathered = torch.empty(world, self._tc.n_params, dtype=torch.float64, device=env.device)

    def _sum_grad_over_ranks(self):
        """The gradient of the last backward pass summed over the ranks into ``_grad``: fp64 per rank, all-gathered,
        summed in rank order and rounded once."""
        import torch.distributed as dist
        self._tc.grad_f64(self._grad64)
        dist.all_gather(list(self._gathered.unbind(0)), self._grad64, group=self.group)
        self._tc.grad_sum_ranks(self._gathered, self._grad)

    def _init_tensor_cores(self):
        env, p, T, N = self.env, self.policy, self.horizon, self.env.num_envs
        check_reference_network(p, env.flat_dim, "tensor_cores=True")
        self._tc = PolicyTrainTC(env, p)
        dev = env.device
        self.last_batch = {"features": torch.empty(T, N, 28, dtype=torch.uint8, device=dev),
                           "counters": torch.empty(T, dtype=torch.int64, device=dev),
                           "actions": torch.empty(T, N, dtype=torch.uint8, device=dev),
                           "logp": torch.empty(T, N, device=dev), "value": torch.empty(T, N, device=dev),
                           "reward": torch.empty(T, N, device=dev), "done": torch.empty(T, N, dtype=torch.bool, device=dev)}
        self._grad = torch.empty(self._tc.n_params, device=dev)
        self._rows = torch.empty(T * N + 1, dtype=torch.int32, device=dev)
        self._iota = torch.arange(T * N, dtype=torch.int32, device=dev)
        self._boot_actions = torch.empty(N, dtype=torch.uint8, device=dev)

    def _sample_tc(self, features: torch.Tensor, actions: torch.Tensor, value: torch.Tensor, logp=None):
        self._ctr += 1
        self._tc.forward_sample(features, self._tc.heads, actions, value=value, logp=logp, noise_scale=0.01 if self.noise else 0.0,
                                counter=self._ctr, seed=self.sample_seed)

    def _collect_tc(self):
        """``horizon`` steps from the current state into ``last_batch`` (features, counters, actions, logp, value, reward,
        done), one ``wab_policy_forward`` launch per step."""
        env, b = self.env, self.last_batch
        for t in range(self.horizon):                                            # :179-189, Policy.forward + select_action
            b["features"][t].copy_(env.last_features)
            self._sample_tc(b["features"][t], b["actions"][t], b["value"][t], b["logp"][t])
            b["counters"][t:t + 1].copy_(self._ctr)
            _, reward, done, _ = env.step(b["actions"][t])
            b["reward"][t].copy_(reward)
            b["done"][t].copy_(done)

    def _train_iteration_tc(self) -> Dict[str, torch.Tensor]:
        env, T, b = self.env, self.horizon, self.last_batch
        if self.mode == "episodic":
            env.reset()
        self._collect_tc()
        log_probs, values = b["logp"].clone().requires_grad_(), b["value"].clone().requires_grad_()
        if self.mode == "episodic":
            loss, info = episodic_actor_critic_loss(log_probs, values, b["reward"], b["done"], self.gamma, self.eps)
        else:
            bootstrap = torch.empty(env.num_envs, device=env.device)
            self._sample_tc(env.last_features, self._boot_actions, bootstrap)
            stats = {}
            if self.group is not None:                                           # normalised over the whole batch
                mean, std = sharding.global_mean_std(horizon_returns(b["reward"], b["done"], bootstrap, self.gamma), self.group)
                stats = {"mean": mean, "std": std, "total_envs": self.total_envs}
            loss, info = horizon_actor_critic_loss(log_probs, values, b["reward"], b["done"], bootstrap, self.gamma, self.eps,
                                                   **stats)
        g_logp, g_value = torch.autograd.grad(loss, [log_probs, values])
        b["g_logp"], b["g_value"] = g_logp, g_value
        # the rows with an upstream gradient, compacted on the device (no host synchronisation): after an env's first
        # done the episodic loss has none
        active = ((g_logp != 0) | (g_value != 0)).reshape(-1)
        pos = torch.cumsum(active, 0, dtype=torch.int32) - 1
        self._rows.scatter_(0, torch.where(active, pos, active.numel()).long(), self._iota)
        n_rows = active.sum(dtype=torch.int64).reshape(1)
        self._tc.backward(b["features"], b["counters"], b["actions"], g_logp, g_value, out=self._grad, rows=self._rows,
                          n_rows=n_rows, noise_scale=0.01 if self.noise else 0.0)
        if self.group is not None:
            self._sum_grad_over_ranks()
        off = 0
        for prm in self.policy.parameters():                                     # .grad = views of the flat gradient
            prm.grad = self._grad[off:off + prm.numel()].view_as(prm)
            off += prm.numel()
        self.optimizer.step()
        self._tc.refresh()
        info.update({"loss": loss.detach(), "mean_reward": b["reward"].mean()})
        return info

    def state_dict(self) -> dict:
        """Environment state (``VecEnv.state_dict``), policy, Adam state, noise counter and sampling seed. With
        ``tensor_cores=True`` (keyed sampling, deterministic gradients) a trainer resumed from it continues bit-exactly.
        In a data-parallel run the env part is this rank's shard; ``sharding.merge_trainer_state_dicts`` joins the ranks'
        dicts, and ``load_state_dict`` takes a merged dict of any layout."""
        return {"env": self.env.state_dict(), "policy": {k: v.detach().cpu().clone() for k, v in self.policy.state_dict().items()},
                "optimizer": copy.deepcopy(self.optimizer.state_dict()), "noise_ctr": int(self._ctr.item()),
                "sample_seed": self.sample_seed}

    def load_state_dict(self, sd: dict):
        self.env.load_state_dict(sd["env"])
        self.policy.load_state_dict(sd["policy"])
        self.optimizer.load_state_dict(sd["optimizer"])
        self._ctr.fill_(int(sd["noise_ctr"]))
        self.sample_seed = int(sd["sample_seed"])
        if self.tensor_cores:
            self._tc.refresh()

    def _observe(self) -> torch.Tensor:
        # gym.spaces.flatten (:188) + np.random.rand(...) / 100 (:189): the keyed kernel the rollout uses
        self.env.flatten_features_noisy(self.env.last_features, self._flat, 0.01 if self.noise else 0.0, self._ctr)
        self._ctr += 1
        return self._flat.clone()        # autograd keeps a reference to the policy input of every step

    def train_iteration(self) -> Dict[str, torch.Tensor]:
        if self.tensor_cores:
            return self._train_iteration_tc()
        env, T = self.env, self.horizon
        if self.mode == "episodic":
            env.reset()                                                          # every env starts an episode (:179)
        log_probs, values, rewards, dones = [], [], [], []
        for _ in range(T):
            probs, value = self.policy(self._observe())
            dist = torch.distributions.Categorical(probs)                        # :114
            action = dist.sample()                                               # :117
            log_probs.append(dist.log_prob(action))                              # :120
            values.append(value.squeeze(1))
            _, reward, done, _ = env.step(action.to(torch.uint8))
            rewards.append(reward.clone())
            dones.append(done.clone())
        log_probs, values = torch.stack(log_probs), torch.stack(values)
        rewards, dones = torch.stack(rewards), torch.stack(dones)
        if self.mode == "episodic":
            loss, info = episodic_actor_critic_loss(log_probs, values, rewards, dones, self.gamma, self.eps)
        else:
            with torch.no_grad():
                _, bootstrap = self.policy(self._observe())                      # critic value of the unfinished tail
            loss, info = horizon_actor_critic_loss(log_probs, values, rewards, dones, bootstrap.squeeze(1), self.gamma, self.eps)
        self.optimizer.zero_grad(set_to_none=True)                               # :159
        loss.backward()                                                          # :165
        self.optimizer.step()
        info.update({"loss": loss.detach(), "mean_reward": rewards.mean()})
        return info
