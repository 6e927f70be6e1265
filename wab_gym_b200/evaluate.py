"""Evaluation of a trained policy on complete episodes, replayable with common random numbers.

The trainers report the mean reward of their own batch: envs that are mid-episode, driven by the sampling policy.
``Evaluator`` answers how good a policy is. It owns a features-only ``VecEnv``, resets it once at construction and keeps
that start state on the device (``VecEnv.save_state``). Every ``evaluate(policy)`` puts the env back to that state,
resets its own draw counter and plays ``episodes_per_env * max_turns`` lockstep steps: ``wab_policy_act`` (the greedy
action, SB3's ``predict(deterministic=True)``) or ``wab_policy_forward`` (the sampled one), then ``VecEnv.step``. Every v1
episode ends by ``max_turns`` (``wab_env.py:328-340``), so every env completes ``episodes_per_env`` episodes and the step
count is fixed. Nothing in the step loop synchronises with the host.

Every draw of the world is keyed by (seed, global env id, episode, site, turn, cell), so episode (n, j) of every call
starts from the same bushes and wolves and sees the same spawn and despawn draws whatever the policy does: two
checkpoints, or two hyper-parameter settings, can be compared episode by episode (common random numbers).

With ``group`` (a ``torch.distributed`` process group) each rank evaluates its contiguous shard of the global env ids
(``sharding.shard_range``) and the results are all-gathered in rank order, so every rank returns the same ``EvalResult``.
Policy draws are keyed by the global env id, so it equals a single-process evaluation of all envs bit for bit, sampled
evaluation included. Every rank must pass the same weights.

``PopulationEvaluator`` scores P policies at once on ``VecEnv(P n, replicas=P)``: every block of n envs repeats the
global ids ``env_id_base ..``, so member p plays exactly the episodes ``Evaluator(n)`` plays, in one launch per step for
all members. With ``group`` rank r owns ``VecEnv(P c_r, replicas=P, env_id_base=env_id_base + first_r)``, its shard
``(first_r, c_r)`` of ``sharding.population_shards(n, W)``, and every rank returns the single-process results bit for bit.
"""
from __future__ import annotations

from typing import Dict, List, NamedTuple, Optional

import torch

from . import sharding
from .policy import Policy, PolicyPopulationTC, PolicyTrunkTC, check_reference_network, stacked_heads
from .vec_env import VecEnv


class EvalResult(NamedTuple):
    """Per-episode results on the host, indexed [env, episode]: episode (n, j) is the j-th episode of global env
    ``env_id_base + n``, played from the same world draws in every evaluation of the same ``Evaluator``."""

    returns: torch.Tensor          # f64[N, k]: the episode's f32 rewards summed in f64, in step order
    lengths: torch.Tensor          # i32[N, k]: steps
    outcome: torch.Tensor          # u8[N, k]: WAB_INFO_OUTCOME of the last step (1 finished, 2 starved, 3 killed)
    eats: torch.Tensor             # i32[N, k]: steps with WAB_INFO_ATE
    first_features: torch.Tensor   # u8[N, k, 28]: the features of the episode's first observation

    def summary(self) -> Dict[str, float]:
        """Mean and (population) standard deviation of the return, mean length, and the fractions of episodes that
        finished (survived to ``max_turns``), starved and were killed."""
        r = self.returns.double().reshape(-1)
        o = self.outcome.reshape(-1)
        n = max(r.numel(), 1)
        return {"episodes": r.numel(), "mean_return": float(r.mean()) if r.numel() else float("nan"),
                "std_return": float(r.std(unbiased=False)) if r.numel() else float("nan"),
                "mean_length": float(self.lengths.double().mean()) if r.numel() else float("nan"),
                "finished": int((o == 1).sum()) / n, "starved": int((o == 2).sum()) / n, "killed": int((o == 3).sum()) / n}


def first_episodes(reward: torch.Tensor, done: torch.Tensor, info: torch.Tensor, k: int):
    """The first ``k`` complete episodes of each env of a [T, N] record (``reward`` f32, ``done`` bool, ``info`` u8 as
    ``VecEnv.step`` returns them): ``(returns f64[N, k], lengths i32[N, k], outcome u8[N, k], eats i32[N, k])`` on the
    record's device. Episode j of env n is the steps after its j-th done up to and including its (j + 1)-th. Raises
    ``ValueError`` if an env completes fewer than ``k`` episodes (one host synchronisation)."""
    if reward.dim() != 2 or tuple(done.shape) != tuple(reward.shape) or tuple(info.shape) != tuple(reward.shape):
        raise ValueError("reward, done and info must be [T, N] tensors of one shape")
    k = int(k)
    if k < 1:
        raise ValueError("k must be >= 1")
    T, N = reward.shape
    dev = reward.device
    d = done.to(torch.bool)
    di = d.to(torch.int64)
    episode = torch.cumsum(di, 0) - di                                   # dones strictly before step t
    complete = di.sum(0)
    if N and int(complete.min()) < k:
        n = int(torch.argmin(complete))
        raise ValueError("env %d completes %d episodes, fewer than k = %d" % (n, int(complete[n]), k))
    cols = torch.arange(N, device=dev)
    slot = episode.clamp(max=k) * N + cols                               # [T, N] into (k + 1) x N; row k takes the rest
    info = info.to(torch.int64)
    lengths = torch.zeros((k + 1) * N, dtype=torch.int64, device=dev).scatter_add_(0, slot.reshape(-1),
                                                                                  torch.ones_like(slot).reshape(-1))
    eats = torch.zeros((k + 1) * N, dtype=torch.int64, device=dev).scatter_add_(0, slot.reshape(-1),
                                                                               ((info >> 2) & 1).reshape(-1))
    outcome = torch.zeros((k + 1) * N, dtype=torch.int64, device=dev).scatter_add_(
        0, slot.reshape(-1), torch.where(d, info & 3, 0).reshape(-1))     # one done per episode: the sum is its outcome
    returns = torch.zeros((k + 1) * N, dtype=torch.float64, device=dev)
    r64 = reward.to(torch.float64)
    for t in range(T):                                                   # EpisodeMonitor's order: one step after another
        returns.index_add_(0, slot[t], r64[t])
    view = lambda x: x.view(k + 1, N)[:k].t().contiguous()
    return view(returns), view(lengths).to(torch.int32), view(outcome).to(torch.uint8), view(eats).to(torch.int32)


def check_policy(policy, flat_dim: int) -> None:
    """What ``tensor_cores=True`` accepts (``policy.check_reference_network``), and a ``ValueError`` too for a module
    that is not shaped like the reference's ``Policy`` at all. Reads shapes and dtypes only."""
    try:
        check_reference_network(policy, flat_dim, "Evaluator")
    except AttributeError as exc:
        raise ValueError("Evaluator is built for the reference's Policy (actor_critic.py:54-97)") from exc


class Evaluator:
    _replicas = 1      # PopulationEvaluator: its members' copies of the env block

    def __init__(self, num_envs: int, game_options: Optional[dict] = None, seed: int = 0, device="cuda",
                 env_id_base: int = 0, episodes_per_env: int = 1, group=None):
        """``num_envs`` environments with global ids ``env_id_base ..`` (with ``group``: over all ranks together),
        ``episodes_per_env`` complete episodes each per evaluation."""
        if int(episodes_per_env) < 1 or int(num_envs) < 1:
            raise ValueError("Evaluator needs num_envs >= 1 and episodes_per_env >= 1")
        self.num_envs, self.episodes_per_env = int(num_envs), int(episodes_per_env)
        self.group = group if sharding._distributed(group) else None
        first, count = 0, self.num_envs
        if self.group is not None:
            import torch.distributed as dist
            first, count = self._shard(dist.get_rank(self.group), dist.get_world_size(self.group))
        self.env = VecEnv(count, game_options=game_options, device=device, seed=seed, env_id_base=int(env_id_base) + first,
                          features=True, emit_grids=False, replicas=self._replicas)
        self.flat_dim, self.n_actions = self.env.flat_dim, self.env.n_actions
        self.max_turns = int(self.env.game_options["max_turns"])
        self.steps = self.episodes_per_env * self.max_turns
        #: the sampling seed of greedy=False: fixed by the env seed, the same on every rank
        self.sample_seed = (int(seed) * 0x9E3779B97F4A7C15 + 0x4556414C) & (2 ** 63 - 1)
        if self.group is not None:
            import torch.distributed as dist
            sig = (self.env.fingerprint, self.num_envs, self.episodes_per_env, int(env_id_base))
            sigs = [None] * dist.get_world_size(self.group)
            dist.all_gather_object(sigs, sig, group=self.group)
            if any(s != sigs[0] for s in sigs):
                raise ValueError("the ranks' Evaluators differ (options, seed, env count or episodes): %r" % (sigs,))
        self.env.reset()
        self._start = self.env.save_state()
        dev, N, T = self.env.device, count, self.steps
        self._ctr = torch.zeros(1, dtype=torch.int64, device=dev)
        self._actions = torch.empty(N, dtype=torch.uint8, device=dev)
        self._reward = torch.empty(T, N, dtype=torch.float32, device=dev)
        self._done = torch.empty(T, N, dtype=torch.bool, device=dev)
        self._info = torch.empty(T, N, dtype=torch.uint8, device=dev)
        self._count = torch.empty(N, dtype=torch.int64, device=dev)
        self._first = torch.empty(self.episodes_per_env + 1, N, 28, dtype=torch.uint8, device=dev)   # row k: later episodes
        self._cols = torch.arange(N, device=dev)
        self._slots = torch.arange(N)
        self._policy = self._tc = self._heads = None

    def _shard(self, rank: int, world: int):
        """(first global id offset, env count) of this rank's handle. Refusals depend on arguments every rank shares, so
        all ranks refuse alike and none waits for a peer."""
        if self.num_envs < world:
            raise ValueError("Evaluator over %d ranks needs at least one env per rank, got %d envs" % (world, self.num_envs))
        return sharding.shard_range(self.num_envs, rank, world)

    def _gather(self, parts):
        """The per-episode tensors of every rank, concatenated in rank order (every rank gets the same)."""
        import torch.distributed as dist
        gathered = [None] * dist.get_world_size(self.group)
        dist.all_gather_object(gathered, parts, group=self.group)
        return gathered

    def restore(self, policy) -> None:
        """Steps 1-3 of ``evaluate``: the start state (one synchronisation), the draw counter, and a copy of ``policy``'s
        weights packed into this evaluator's own buffers (``policy`` itself is only read)."""
        check_policy(policy, self.flat_dim)
        A = policy.action_head.out_features
        if self._policy is None or self._policy.action_head.out_features != A:
            with torch.random.fork_rng(devices=[]):                     # the initialisation draws stay off the global RNG
                self._policy = Policy(self.flat_dim, A).to(self.env.device)
            self._tc = PolicyTrunkTC(self.env, self._policy)
        with torch.no_grad():
            for name in ("affine1", "affine2", "affine3", "action_head", "value_head"):
                mine, theirs = getattr(self._policy, name), getattr(policy, name)
                mine.weight.copy_(theirs.weight.detach())
                mine.bias.copy_(theirs.bias.detach())
        self._tc.refresh()
        self._heads = stacked_heads(self._policy)
        self._rewind()

    def _rewind(self) -> None:
        self.env.load_state(self._start, slots=self._slots)
        self._ctr.zero_()

    def _act(self, greedy: bool, scale: float) -> None:
        """One step's actions into ``self._actions``: the one launch of the step loop that depends on the policy."""
        if greedy:
            self._tc.forward_greedy(self.env.last_features, self._heads, self._actions, noise_scale=scale, counter=self._ctr)
        else:
            self._tc.forward_sample(self.env.last_features, self._heads, self._actions, noise_scale=scale, counter=self._ctr,
                                    seed=self.sample_seed)

    @torch.no_grad()
    def play(self, greedy: bool = True, noise: bool = True):
        """Step 4 of ``evaluate``: ``steps`` lockstep steps of the restored policy. Returns the device record
        ``(reward f32[T, N], done bool[T, N], info u8[T, N])`` (buffers reused by the next call). Nothing here
        synchronises with the host."""
        if self._tc is None:
            raise RuntimeError("play() follows restore(policy)")
        env, k = self.env, self.episodes_per_env
        scale = 0.01 if noise else 0.0
        self._count.zero_()
        self._first[0].copy_(env.last_features)
        for t in range(self.steps):
            self._ctr += 1
            self._act(greedy, scale)
            _, reward, done, info = env.step(self._actions)
            self._reward[t].copy_(reward)
            self._done[t].copy_(done)
            self._info[t].copy_(info["info"])
            # the first observation of the next episode (auto-reset) goes to row min(episodes so far, k); others to row k
            self._count += done
            self._first[torch.where(done, self._count.clamp(max=k), k), self._cols] = env.last_features
        return self._reward, self._done, self._info

    def evaluate(self, policy, greedy: bool = True, noise: bool = True) -> EvalResult:
        """Play ``episodes_per_env`` complete episodes per env with ``policy`` from the saved start state: the greedy
        action (``greedy=True``) or the sampled one, with the reference's ``U/100`` input noise (``noise=True``) or
        without. Returns the per-episode results on the host, the same on every rank. ``policy`` (any device) and any
        trainer that owns it are left untouched."""
        self.restore(policy)
        parts = self._episodes(*self.play(greedy, noise))
        if self.group is not None:
            gathered = self._gather(parts)
            parts = [torch.cat([g[i] for g in gathered]) for i in range(len(parts))]
        return EvalResult(*parts)

    def _episodes(self, reward, done, info):
        """The five per-episode tensors of ``EvalResult`` of the record ``play`` left, on the host."""
        returns, lengths, outcome, eats = first_episodes(reward, done, info, self.episodes_per_env)
        first = self._first[:self.episodes_per_env].transpose(0, 1).contiguous()
        return [t.cpu() for t in (returns, lengths, outcome, eats, first)]

    def close(self):
        self.env.close()


class PopulationEvaluator(Evaluator):
    """P policies scored on the same episodes in one launch per step. It owns ``VecEnv(P n, replicas=P)``: block p of n
    envs replays the world draws of ``Evaluator(n, ...)``'s envs, member p acts on it through its row block of one
    ``PolicyPopulationTC`` (``wab_policy_act_population`` or ``wab_policy_forward_population``), and every policy draw
    is keyed as that evaluator keys it. So ``evaluate(policies)[p]`` equals ``Evaluator(n, game_options, seed, env_id_base,
    episodes_per_env).evaluate(policies[p])`` bit for bit, and the P results line up episode by episode (common random
    numbers: what separates close policies such as the members of a population-based training run). ``envs_per_member``
    = n is a multiple of 128, 1 <= ``members`` <= 64.

    With ``group`` (W > 1 ranks) rank r owns ``VecEnv(P c_r, replicas=P, env_id_base=env_id_base + first_r)`` for its shard
    ``(first_r, c_r)`` of ``sharding.population_shards(n, W)`` (each c_r a positive multiple of 128). Member p's per-episode
    tensors are all-gathered in rank order, so every rank returns the single-process ``results`` bit for bit. Every rank
    must pass the same policies."""

    def __init__(self, members: int, envs_per_member: int, game_options: Optional[dict] = None, seed: int = 0,
                 device="cuda", env_id_base: int = 0, episodes_per_env: int = 1, group=None):
        P, n = int(members), int(envs_per_member)
        group = sharding.process_group(group, "PopulationEvaluator")
        if not 1 <= P <= 64:
            raise ValueError("a population has 1 to 64 members")
        if n < 128 or n % 128 != 0:
            raise ValueError("PopulationEvaluator needs envs_per_member a positive multiple of 128, got %d" % n)
        self.members, self.envs_per_member, self._replicas = P, n, P
        super().__init__(P * n, game_options=game_options, seed=seed, device=device, env_id_base=env_id_base,
                         episodes_per_env=episodes_per_env, group=group)
        self.shard_envs = self.env.num_envs // P         # c_r: this rank's envs of each member
        self._policies = None

    def _shard(self, rank: int, world: int):
        first, c = sharding.population_shards(self.envs_per_member, world)[rank]
        return first, self.members * c

    def restore(self, policies) -> None:
        """``Evaluator.restore`` for P policies: each one's weights copied into this evaluator's own member and packed."""
        policies = list(policies)
        if len(policies) != self.members:
            raise ValueError("evaluate needs one policy per member (%d), got %d" % (self.members, len(policies)))
        for pol in policies:
            check_policy(pol, self.flat_dim)
        A = policies[0].action_head.out_features
        if any(pol.action_head.out_features != A for pol in policies):
            raise ValueError("every member of a population has the same action count")
        if self._policies is None or self._tc.n_actions != A:
            with torch.random.fork_rng(devices=[]):                     # the initialisation draws stay off the global RNG
                self._policies = [Policy(self.flat_dim, A).to(self.env.device) for _ in range(self.members)]
            self._tc = PolicyPopulationTC(self.env, self._policies)
        with torch.no_grad():
            for mine, theirs in zip(self._policies, policies):
                for a, b in zip(mine.parameters(), theirs.parameters()):
                    a.copy_(b.detach())
        self._tc.refresh()
        self._rewind()

    def _act(self, greedy: bool, scale: float) -> None:
        # the buffers are this evaluator's own and restore() packed every member: the launch alone
        self._tc._launch(None if greedy else self.sample_seed, self.env.last_features, self._actions, None, None, None, None,
                         scale, self._ctr, 0.01)

    def evaluate(self, policies, greedy: bool = True, noise: bool = True) -> List[EvalResult]:
        """``Evaluator.evaluate`` of every member at once: ``results[p]`` is ``policies[p]``'s ``EvalResult`` over the n
        envs of block p, whose global ids ``env_id_base ..`` are the same in every block. The policies are only read."""
        self.restore(policies)
        parts = self._episodes(*self.play(greedy, noise))
        P = self.members
        if self.group is None:
            split = [t.view(P, self.envs_per_member, *t.shape[1:]) for t in parts]
        else:                                            # member p: its c_r rows of every rank, in rank order
            gathered = self._gather(parts)
            split = [torch.cat([g[i].view(P, -1, *g[i].shape[1:]) for g in gathered], dim=1) for i in range(len(parts))]
        return [EvalResult(*(t[p] for t in split)) for p in range(P)]
