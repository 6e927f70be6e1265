"""A population of PPO policies trained side by side: hyper-parameter sweeps, seeds for error bars and the primitives of
population-based training, on one environment handle and one launch per kernel for all members.

``PPOPopulation`` trains P members (1 <= P <= 64) on ONE features-enabled ``VecEnv`` of N = P n envs, n a multiple of 128.
Member p owns env rows [p n, (p + 1) n), i.e. global env ids ``env_id_base + p n + j``. Every draw of the environment and
of the policy is keyed by the global env id, and the population kernels give each member's tiles to its CTAs in the
order a single-policy launch uses, so member p is bit for bit the run ``PPOTrainer(VecEnv(n, env_id_base=p n), ...)``
would produce alone with the same policy, hyper-parameters and sampling seed: its batch, weights, Adam state and
diagnostics. A sweep run as a population gives the same results as the sweep run one member at a time, and
``Evaluator.evaluate(pop.policies[p])`` compares members on identical episodes.

Per iteration (``PPOTrainer``'s, for all members at once): ``horizon`` collection steps of one
``wab_policy_forward_population`` launch and one env step each, one more forward for the bootstrap, GAE over [T, N] with
per-column gamma and gamma lam, advantage normalisation per member, then ``epochs`` passes over one shared permutation of
member-local rows (seeded as ``PPOTrainer`` seeds it), translated to each member's global rows, cut into ``minibatches``
slices. Each slice is ONE ``wab_policy_ppo_backward_population`` launch, then a global-norm clip and an Adam step per
member. Every per-member statistic (normalisation mean and std, gradient norm, mean reward, diagnostics) is computed on a
contiguous tensor of that member alone, as ``PPOTrainer`` computes it, so it rounds the same way. Nothing in an iteration
synchronises with the host.

Data-parallel populations (``group``, a ``torch.distributed`` process group of W > 1 ranks): every rank holds all P
members, each on its contiguous shard ``[first_r, first_r + c_r)`` of the member's n envs (``sharding.population_shards``,
c_r a positive multiple of 128), on ONE handle ``VecEnv(P c_r, env_id_base=B + first_r, blocks=P, block_stride=n)``: row
p c_r + j is member p's global id ``B + p n + first_r + j``, the id it has in a single-process population whose first id is
B. Construction all-gathers each rank's layout and signature, checks them on every rank (so a refusal is raised on every
rank and none is left waiting in a collective), then broadcasts rank 0's policies and sampling seed. Per iteration each
member does what ``PPOTrainer(group)`` does: advantages normalised by the member's mean and std over all ranks
(``sharding.global_mean_std_members``: two collectives for all members), one permutation per member seeded with the first
global id of its shard on this rank, minibatch k's weights divided by its row count summed over the ranks, and after each
population backward the fp64 gradient of every member (``wab_policy_backward_population_grad_f64``) all-gathered once and
summed in rank order (``wab_policy_grad_sum_ranks``) before the clip and Adam. So every rank holds bit-identical weights,
Adam state and hyper-parameters, and member p is bit for bit the 1-member data-parallel population on ids from B + p n.
Collection is invariant to the world size; training, like that of the data-parallel trainers, is not (``a2c``'s module
docstring), but ``sharding.merge_population_state_dicts`` of the ranks' ``state_dict()``s resumes on any layout. A group of
one rank is the single-process population.
"""
from __future__ import annotations

import copy
import inspect
from typing import Dict, List, Optional

import torch

from . import sharding
from .policy import Policy, PolicyPopulationTC, check_reference_network
from .ppo import PPOTrainer, _perm_seed, gae, ppo_loss
from .vec_env import STATE_FORMAT, EnvStates, VecEnv

#: the per-member hyper-parameters and their defaults (``PPOTrainer``'s)
HYPERPARAMETERS = {k: inspect.signature(PPOTrainer.__init__).parameters[k].default
                   for k in ("lr", "gamma", "lam", "clip_eps", "vf_coef", "ent_coef", "max_grad_norm")}


def member_hyperparameters(hyperparameters, n_members: int) -> List[Dict[str, float]]:
    """The P complete hyper-parameter dicts: a missing key takes ``PPOTrainer``'s default. Raises ``ValueError`` for a
    list of another length, an unknown key, or a value ``PPOTrainer`` refuses (clip_eps or max_grad_norm <= 0)."""
    if hyperparameters is None:
        hyperparameters = [{} for _ in range(n_members)]
    hyperparameters = list(hyperparameters)
    if len(hyperparameters) != n_members:
        raise ValueError("hyperparameters must hold one dict per member (%d), got %d" % (n_members, len(hyperparameters)))
    out = []
    for p, hp in enumerate(hyperparameters):
        unknown = set(hp) - set(HYPERPARAMETERS)
        if unknown:
            raise ValueError("member %d: unknown hyper-parameter(s) %s; known: %s" % (p, sorted(unknown), sorted(HYPERPARAMETERS)))
        full = {k: float(hp.get(k, d)) for k, d in HYPERPARAMETERS.items()}
        if not full["clip_eps"] > 0 or not full["max_grad_norm"] > 0:
            raise ValueError("member %d: clip_eps and max_grad_norm must be > 0" % p)
        out.append(full)
    return out


def member_rows(perm: torch.Tensor, n_members: int, member_envs: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Member-local rows t n + j (``perm``: int32[M], shared by every member, or int32[P, M], one list per member) -> each
    member's global rows t N + p n + j, N = P n: int32[P, M] (written into ``out`` when given, which may be a column slice
    of a wider buffer)."""
    n = member_envs
    local = (perm // n) * (n_members * n) + perm % n
    if local.dim() == 1:
        local = local[None, :]
    offsets = torch.arange(n_members, dtype=perm.dtype, device=perm.device) * n
    if out is None:
        return local + offsets[:, None]
    return torch.add(local, offsets[:, None], out=out)


class PPOPopulation:
    """P ``PPOTrainer`` runs in one: see the module docstring. ``members`` = P; ``policies`` (optional) = P reference
    ``Policy`` modules (fresh ones otherwise); ``hyperparameters`` = P dicts over ``HYPERPARAMETERS`` (missing keys take
    ``PPOTrainer``'s defaults). ``horizon``, ``epochs``, ``minibatches``, ``noise`` and the sampling seed are shared."""

    def __init__(self, env: VecEnv, members: int, hyperparameters=None, policies=None, horizon: int = 64, epochs: int = 4,
                 minibatches: int = 4, noise: bool = True, group=None):
        # everything PPOTrainer refuses before any device work; with a group, on every rank (the layout is checked too)
        self.group = sharding.process_group(group, "PPOPopulation")
        if self.group is None:
            policies = self._validate(env, members, hyperparameters, policies, horizon, epochs, minibatches, True)
        else:
            policies = self._join_layout(env, members, hyperparameters, policies, horizon, epochs, minibatches, noise)
        P, N, n = int(members), env.num_envs, env.num_envs // int(members)
        if policies is None:
            policies = [Policy(env.flat_dim, env.n_actions) for _ in range(P)]
        self.env, self.n_members, self.member_envs = env, P, n
        self.horizon, self.epochs, self.minibatches, self.noise = int(horizon), int(epochs), int(minibatches), noise
        self.policies = [pol.to(env.device) for pol in policies]
        self.optimizers = [torch.optim.Adam(pol.parameters(), lr=hp["lr"]) for pol, hp in zip(self.policies, self.hyperparameters)]
        self._ctr = torch.zeros(1, dtype=torch.int64, device=env.device)
        self.sample_seed = int(torch.initial_seed()) & (2 ** 63 - 1)
        self.iteration = 0
        self._tc = PolicyPopulationTC(env, self.policies)
        T, dev = self.horizon, env.device
        self.last_batch = {"features": torch.empty(T, N, 28, dtype=torch.uint8, device=dev),
                           "counters": torch.empty(T, dtype=torch.int64, device=dev),
                           "actions": torch.empty(T, N, dtype=torch.uint8, device=dev),
                           "logp": torch.empty(T, N, device=dev), "value": torch.empty(T, N, device=dev),
                           "reward": torch.empty(T, N, device=dev), "done": torch.empty(T, N, dtype=torch.bool, device=dev),
                           "bootstrap": torch.empty(N, device=dev), "advantage": torch.empty(T, N, device=dev),
                           "target": torch.empty(T, N, device=dev)}
        self._boot_actions = torch.empty(N, dtype=torch.uint8, device=dev)
        self._new = {k: torch.empty(T, N, device=dev) for k in ("logp", "value", "entropy")}
        # one permutation of member-local rows per epoch, shared by the members (single process) or one per member (group)
        self._perm = torch.empty(T * n if self.group is None else (P, T * n), dtype=torch.int32, device=dev)
        self._bounds = sharding.minibatch_bounds(T * n, self.minibatches)
        # the row count minibatch k's weights are divided by: this process's, or the sum over the ranks
        self._global_counts = ([self._bounds[k + 1] - self._bounds[k] for k in range(self.minibatches)] if self.group is None
                               else sharding.global_minibatch_counts([T * c for c in self._shard_counts], self.minibatches))
        # minibatch k's row lists [P][M_k], M_k rounded up to 64 entries so that each member's gathered rows start 256-byte
        # aligned (a contiguous tensor of its own, like PPOTrainer's); the padding entries are never read by the kernel
        sizes = [self._bounds[k + 1] - self._bounds[k] for k in range(self.minibatches)]
        self._mb_rows = [torch.zeros(P, (m + 63) // 64 * 64, dtype=torch.int32, device=dev) for m in sizes]
        self._mb_counts = [torch.full((P,), m, dtype=torch.int64, device=dev) for m in sizes]
        self._grad = torch.zeros(P, self._tc.grad_stride, device=dev)
        n_params = self._tc.n_params
        for p, pol in enumerate(self.policies):          # .grad = views of member p's row of the gradient
            off = 0
            for prm in pol.parameters():
                prm.grad = self._grad[p, off:off + prm.numel()].view_as(prm)
                off += prm.numel()
            assert off == n_params
        self._set_discounts()
        env.reset()
        if self.group is not None:
            self._join_weights()

    def _validate(self, env, members, hyperparameters, policies, horizon, epochs, minibatches, single: bool):
        """The constructor's refusals (``ValueError``), before any device work. Sets ``hyperparameters``; returns the
        policies as a list (or None)."""
        P, N = int(members), env.num_envs
        if not 1 <= P <= 64:
            raise ValueError("a population has 1 to 64 members")
        if N % P != 0 or (N // P) % 128 != 0:
            raise ValueError("PPOPopulation needs num_envs = members * n with n a multiple of 128 (got %d envs, %d members)" % (N, P))
        if not env.with_features:
            raise ValueError("PPOPopulation needs VecEnv(features=True)")
        if getattr(env, "replicas", 1) > 1:
            raise ValueError("PPOPopulation refuses a VecEnv with replicas: its members own distinct env ids")
        n = N // P
        blocks, stride = getattr(env, "blocks", 1), getattr(env, "block_stride", 0)
        if single and not (blocks == 1 or (blocks == P and stride == n)):
            raise ValueError("a single-process PPOPopulation needs a plain VecEnv (or blocks=%d, block_stride=%d: the same ids)"
                             % (P, n))
        if epochs < 1 or minibatches < 1 or int(horizon) * n < minibatches:
            raise ValueError("PPOPopulation needs epochs >= 1 and 1 <= minibatches <= horizon * n")
        self.hyperparameters = member_hyperparameters(hyperparameters, P)
        if policies is None:
            return None
        policies = list(policies)
        if len(policies) != P:
            raise ValueError("policies must hold one Policy per member (%d), got %d" % (P, len(policies)))
        for pol in policies:
            check_reference_network(pol, env.flat_dim, "PPOPopulation")
        if any(pol.action_head.out_features != env.n_actions for pol in policies):
            raise ValueError("every member's action head must have the environment's %d actions" % env.n_actions)
        return policies

    def _signature(self, env, members, horizon, epochs, minibatches, noise) -> tuple:
        """What every rank of a data-parallel population must agree on."""
        return (int(env.fingerprint), int(env.n_actions), int(members), int(horizon), int(epochs), int(minibatches), bool(noise),
                tuple(tuple(sorted(hp.items())) for hp in self.hyperparameters))

    def _join_layout(self, env, members, hyperparameters, policies, horizon, epochs, minibatches, noise):
        """The refusals of a data-parallel population on every rank: this rank's own checks (an exception of any type is a
        refusal), then one all-gather of every rank's verdict, layout and signature (one host synchronisation), then the
        layout check. Any refusal raises ``ValueError`` on every rank."""
        import torch.distributed as dist
        err, sig, local = None, None, None
        try:
            policies = self._validate(env, members, hyperparameters, policies, horizon, epochs, minibatches, False)
            sig = self._signature(env, members, horizon, epochs, minibatches, noise)
        except Exception as exc:          # any refusal, of any type, is gathered: no rank skips the collective below
            local = exc
            err = str(exc) if isinstance(exc, ValueError) else "%s: %s" % (type(exc).__name__, exc)
        info = (int(env.env_id_base), int(env.num_envs), int(getattr(env, "blocks", 1)), int(getattr(env, "block_stride", 0)),
                sig, err)
        infos = [None] * dist.get_world_size(self.group)
        dist.all_gather_object(infos, info, group=self.group)
        for r, i in enumerate(infos):
            if i[5] is not None:
                raise ValueError("rank %d refused the population: %s" % (r, i[5])) from local
        self.first_id, self.total_member_envs = sharding.check_population_shards([i[:5] for i in infos], int(members))
        self._shard_counts = [int(i[1]) // int(members) for i in infos]
        return policies

    def _join_weights(self):
        """Rank 0's policies and sampling seed on every rank, and the buffers of the cross-rank gradient sum."""
        import torch.distributed as dist
        dev, world = self.env.device, dist.get_world_size(self.group)
        src = dist.get_global_rank(self.group, 0)
        with torch.no_grad():
            for pol in self.policies:
                for prm in pol.parameters():
                    dist.broadcast(prm.data, src, group=self.group)
        seed = torch.tensor([self.sample_seed], dtype=torch.int64, device=dev)
        dist.broadcast(seed, src, group=self.group)
        self.sample_seed = int(seed.item())
        self._tc.refresh()
        self._grad64 = torch.empty(self.n_members, self._tc.grad_stride, dtype=torch.float64, device=dev)
        self._gathered = torch.empty(world, self.n_members, self._tc.grad_stride, dtype=torch.float64, device=dev)

    def _member_first_id(self, p: int) -> int:
        """The global id of member p's first row on this handle."""
        return int(self.env.global_ids([p * self.member_envs])[0])

    def _sum_grad_over_ranks(self):
        """Every member's gradient of the last population backward summed over the ranks into ``_grad``: fp64 per rank,
        one all-gather of [P, stride], summed in rank order and rounded once."""
        import torch.distributed as dist
        self._tc.grad_f64(self._grad64)
        dist.all_gather(list(self._gathered.unbind(0)), self._grad64, group=self.group)
        self._tc.grad_sum_ranks(self._gathered, self._grad)

    def _set_discounts(self):
        """The per-column gamma and gamma * lam of GAE: member p's values on its n columns (gamma * lam in double, rounded
        once to fp32, as ``gae`` rounds a float gamma * lam)."""
        n, dev = self.member_envs, self.env.device
        self._gamma = torch.tensor([hp["gamma"] for hp in self.hyperparameters], dtype=torch.float32).repeat_interleave(n).to(dev)
        self._gamma_lam = torch.tensor([hp["gamma"] * hp["lam"] for hp in self.hyperparameters],
                                       dtype=torch.float32).repeat_interleave(n).to(dev)

    def _sample(self, features: torch.Tensor, actions: torch.Tensor, value: torch.Tensor, logp=None):
        self._ctr += 1
        self._tc.forward_sample(features, actions, value=value, logp=logp, noise_scale=0.01 if self.noise else 0.0,
                                counter=self._ctr, seed=self.sample_seed)

    def _collect(self):
        env, b = self.env, self.last_batch
        for t in range(self.horizon):
            b["features"][t].copy_(env.last_features)
            self._sample(b["features"][t], b["actions"][t], b["value"][t], b["logp"][t])
            b["counters"][t:t + 1].copy_(self._ctr)
            _, reward, done, _ = env.step(b["actions"][t])
            b["reward"][t].copy_(reward)
            b["done"][t].copy_(done)

    def _by_member(self, x: torch.Tensor) -> torch.Tensor:
        """[T, N] -> [P, T, n], contiguous: member p's columns as the [T, n] tensor a standalone trainer holds."""
        T = x.shape[0]
        return x.view(T, self.n_members, self.member_envs).transpose(0, 1).contiguous()

    def train_iteration(self) -> Dict[str, torch.Tensor]:
        """One PPO iteration of every member. Returns device tensors: for each ``ppo_loss`` diagnostic and ``grad_norm``,
        [P, epochs * minibatches] (member p's row is what its ``PPOTrainer.train_iteration`` returns), and
        ``mean_reward`` [P]."""
        env, b, P, n = self.env, self.last_batch, self.n_members, self.member_envs
        T, N, hps = self.horizon, env.num_envs, self.hyperparameters
        noise = 0.01 if self.noise else 0.0
        self._collect()
        self._sample(env.last_features, self._boot_actions, b["bootstrap"])
        adv, ret = gae(b["reward"], b["done"], b["value"], b["bootstrap"], self._gamma, None, gamma_lam=self._gamma_lam)
        b["target"].copy_(ret)
        by_member = self._by_member(adv)
        if self.group is None:
            mean = torch.stack([by_member[p].mean() for p in range(P)])
            std = torch.stack([by_member[p].std() for p in range(P)])
        else:
            mean, std = sharding.global_mean_std_members(by_member, self.group)
        by_member.sub_(mean[:, None, None]).div_((std + 1e-8)[:, None, None])   # normalised once per member's batch
        b["advantage"].view(T, P, n).copy_(by_member.transpose(0, 1))
        del adv, ret, by_member
        flat = {k: b[k].view(-1) for k in ("logp", "advantage", "target")}
        new = {k: v.view(-1) for k, v in self._new.items()}
        stats = [[] for _ in range(P)]
        first_ids = None if self.group is None else [self._member_first_id(p) for p in range(P)]
        for epoch in range(self.epochs):
            if self.group is None:
                gen = torch.Generator(device=env.device)
                gen.manual_seed(_perm_seed(self.sample_seed, self.iteration, epoch))
                torch.randperm(self._perm.numel(), generator=gen, out=self._perm)
            else:                                        # member p's shard shuffled as its data-parallel trainer would
                for p in range(P):
                    gen = torch.Generator(device=env.device)
                    gen.manual_seed(_perm_seed(self.sample_seed, self.iteration, epoch, first_ids[p]))
                    torch.randperm(self._perm.shape[1], generator=gen, out=self._perm[p])
            for k in range(self.minibatches):
                m = self._bounds[k + 1] - self._bounds[k]
                rows = self._mb_rows[k]
                member_rows(self._perm[..., self._bounds[k]:self._bounds[k + 1]], P, n, out=rows[:, :m])
                mg = self._global_counts[k]
                coefs = [(hp["clip_eps"], 1.0 / mg, hp["vf_coef"] / mg, hp["ent_coef"] / mg) for hp in hps]
                self._tc.ppo_backward(b["features"], b["counters"], b["actions"], b["logp"], b["advantage"], b["target"],
                                      rows, self._mb_counts[k], coefs, out=self._grad, logp=self._new["logp"],
                                      value=self._new["value"], entropy=self._new["entropy"], noise_scale=noise)
                if self.group is not None:
                    self._sum_grad_over_ranks()
                picked = [t.index_select(0, rows.view(-1)).view(P, -1) for t in (new["logp"], new["value"], new["entropy"],
                                                                                   flat["logp"], flat["advantage"], flat["target"])]
                for p, hp in enumerate(hps):
                    grad = self._grad[p, :self._tc.n_params]
                    norm = torch.linalg.vector_norm(grad)
                    grad.mul_(torch.clamp(hp["max_grad_norm"] / (norm + 1e-6), max=1.0))
                    self.optimizers[p].step()
                    _, info = ppo_loss(*(t[p, :m] for t in picked), hp["clip_eps"], hp["vf_coef"], hp["ent_coef"])
                    info["grad_norm"] = norm
                    stats[p].append(info)
        self.iteration += 1
        out = {key: torch.stack([torch.stack([s[key] for s in stats[p]]) for p in range(P)]) for key in stats[0][0]}
        reward = self._by_member(b["reward"])
        out["mean_reward"] = torch.stack([reward[p].mean() for p in range(P)])
        return out

    # ------------------------------------------------------------------ state
    def state_dict(self) -> dict:
        """The env, every member's policy, Adam state and hyper-parameters, the noise counter, the sampling seed and the
        iteration: a population resumed from it continues bit for bit."""
        return {"env": self.env.state_dict(),
                "policies": [{k: v.detach().cpu().clone() for k, v in pol.state_dict().items()} for pol in self.policies],
                "optimizers": [copy.deepcopy(opt.state_dict()) for opt in self.optimizers],
                "hyperparameters": copy.deepcopy(self.hyperparameters), "noise_ctr": int(self._ctr.item()),
                "sample_seed": self.sample_seed, "iteration": self.iteration}

    def load_state_dict(self, sd: dict):
        if len(sd["policies"]) != self.n_members:
            raise ValueError("the state dict holds %d members, this population %d" % (len(sd["policies"]), self.n_members))
        self.hyperparameters = member_hyperparameters(sd["hyperparameters"], self.n_members)
        self.env.load_state_dict(sd["env"])
        for pol, opt, psd, osd in zip(self.policies, self.optimizers, sd["policies"], sd["optimizers"]):
            pol.load_state_dict(psd)
            opt.load_state_dict(osd)
        self._ctr.fill_(int(sd["noise_ctr"]))
        self.sample_seed = int(sd["sample_seed"])
        self.iteration = int(sd["iteration"])
        self._set_discounts()
        self._tc.refresh()

    def set_member_hyperparameters(self, p: int, hp: Dict[str, float]):
        """Member p's hyper-parameters: the keys of ``hp`` replace p's (the others stay), validated as the constructor
        validates them, and written everywhere they live: the dict, the lr of p's Adam and the GAE discounts. (After
        ``load_member_state_dict(p, member_state_dict(q))`` p's Adam holds q's lr, so this is the explore step of
        population-based training.)"""
        self._member_slots(p)
        full = member_hyperparameters([{**self.hyperparameters[p], **hp}], 1)[0]
        self.hyperparameters[p] = full
        for group in self.optimizers[p].param_groups:
            group["lr"] = full["lr"]
        self._set_discounts()

    def _member_slots(self, p: int) -> torch.Tensor:
        if not 0 <= p < self.n_members:
            raise ValueError("member %d of %d" % (p, self.n_members))
        return torch.arange(p * self.member_envs, (p + 1) * self.member_envs, dtype=torch.int64)

    def member_state_dict(self, p: int) -> dict:
        """Member p as a ``PPOTrainer`` state dict: ``PPOTrainer.load_state_dict`` on ``VecEnv(n, env_id_base=p n)`` (this
        env's options and seed) continues exactly as member p would. The env part holds member p's envs (and, for member
        0, the statistics totals of the whole handle); ``hyperparameters`` is member p's dict, for
        ``load_member_state_dict``."""
        st = self.env.save_state(self._member_slots(p))
        stats = self.env.state_dict()["stats"] if p == 0 else torch.zeros(8, dtype=torch.int64)
        return {"env": {"format": STATE_FORMAT, "fingerprint": st.fingerprint, "env_ids": st.env_ids.clone(),
                        "records": st.records.cpu(), "stats": stats},
                "policy": {k: v.detach().cpu().clone() for k, v in self.policies[p].state_dict().items()},
                "optimizer": copy.deepcopy(self.optimizers[p].state_dict()), "hyperparameters": dict(self.hyperparameters[p]),
                "noise_ctr": int(self._ctr.item()), "sample_seed": self.sample_seed, "iteration": self.iteration}

    def load_member_state_dict(self, p: int, sd: dict):
        """The inverse of ``member_state_dict``: member p takes the policy, the Adam state and (when present) the
        hyper-parameters of ``sd``. Its envs take the env part only when that holds member p's own env ids (a dict of
        member p, or of a ``PPOTrainer`` on its ids); the dict of another member q leaves them where they are, which makes
        ``load_member_state_dict(p, member_state_dict(q))`` the "exploit" step of population-based training. The noise
        counter, sampling seed and iteration are the population's and are not changed."""
        slots = self._member_slots(p)
        ids = torch.as_tensor(sd["env"]["env_ids"], dtype=torch.int64).reshape(-1)
        own_ids = self.env.global_ids(slots)             # contiguous: member p's shard of ids on this handle
        own = ids.numel() == slots.numel() and torch.equal(torch.sort(ids).values, own_ids)
        hp = member_hyperparameters([sd.get("hyperparameters", self.hyperparameters[p])], 1)[0]
        if own:
            records = sharding.select_shard_records(sd["env"], int(own_ids[0]), self.member_envs,
                                                    self.env.fingerprint, self.env.record_bytes, STATE_FORMAT)
            self.env.load_state(EnvStates(records, own_ids, self.env.fingerprint))
        self.policies[p].load_state_dict(sd["policy"])
        self.optimizers[p].load_state_dict(sd["optimizer"])
        self.hyperparameters[p] = hp
        self._set_discounts()
        self._tc.refresh([p])
