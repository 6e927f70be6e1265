"""Population-based training (Jaderberg et al. 2017, "Population Based Training of Neural Networks"), truncation selection,
over a ``PPOPopulation`` scored by a ``PopulationEvaluator``.

``PopulationBasedTraining.step()`` runs one ``train_iteration()`` of every member. After every ``interval``-th iteration
it runs a ready event:

1. fitness: each member's mean evaluation return (f64), every member played on the same episodes (common random
   numbers, ``PopulationEvaluator``), so the ranking is not decided by which worlds a member happened to draw;
2. rank the members by fitness, highest first, ties to the lower index;
3. exploit: each of the bottom ``floor(fraction P)`` members p copies a source q drawn from the top ``floor(fraction P)``
   (``load_member_state_dict(p, member_state_dict(q))``): p keeps its own envs and takes q's policy, Adam state and
   hyper-parameters;
4. explore: each key of ``perturb`` of p is multiplied by a factor drawn from ``factors``
   (``PPOPopulation.set_member_hyperparameters``, which keeps Adam's lr and the GAE discounts in step with the dict).

Every draw is keyed by (seed, iteration, member, site) through ``ppo._seed``, never by a global generator, so a ready
event can be replayed from its iteration, and ``state_dict()`` resumes a run bit for bit.
"""
from __future__ import annotations

import copy
import math
from typing import Dict, List, Sequence, Tuple

import torch

from .ppo import _seed

#: the hyper-parameters a ready event may perturb: any positive factor keeps them valid. gamma and lam are discounts in
#: [0, 1], which a factor above 1 could leave.
PERTURBABLE = ("lr", "clip_eps", "vf_coef", "ent_coef", "max_grad_norm")


def rank_members(fitness: Sequence[float]) -> List[int]:
    """Member indices by fitness, highest first; equal fitness goes to the lower index first."""
    return sorted(range(len(fitness)), key=lambda p: (-float(fitness[p]), p))


def truncation(ranking: Sequence[int], fraction: float) -> Tuple[List[int], List[int]]:
    """``(bottom, top)``: the last and the first ``floor(fraction P)`` entries of ``ranking``."""
    k = math.floor(float(fraction) * len(ranking))
    return list(ranking[len(ranking) - k:]) if k else [], list(ranking[:k])


def draw_source(seed: int, iteration: int, member: int, top: Sequence[int]) -> int:
    """The member of ``top`` that ``member`` copies at the ready event after ``iteration``."""
    return top[_seed(seed, iteration, member, 0) % len(top)]


def draw_factor(seed: int, iteration: int, member: int, key: str, factors: Sequence[float]) -> float:
    """The factor ``member``'s hyper-parameter ``key`` is multiplied by at the ready event after ``iteration``. The site is
    the key's place in ``PERTURBABLE``, so a key's draw does not depend on which other keys are perturbed."""
    return float(factors[_seed(seed, iteration, member, 1 + PERTURBABLE.index(key)) % len(factors)])


class PopulationBasedTraining:
    """Population-based training of ``population`` (a ``PPOPopulation``) scored by ``evaluator`` (a ``PopulationEvaluator``
    with the same member count): see the module docstring. ``greedy`` selects the evaluator's greedy or sampled actions.
    ``history`` holds one dict per ready event: ``iteration``, ``fitness`` (f64[P]), ``ranking``, ``copies`` [(p, q)],
    ``factors`` {p: {key: factor}} and ``hyperparameters`` (every member's, after the event).

    A data-parallel population and evaluator (the same ``group``) work unchanged: every rank holds every member, the
    evaluator returns the same fitness on every rank, and the keyed draws are the same there, so every rank takes the same
    decisions and no member state moves between ranks. ``state_dict()`` is then per rank; its ``population`` parts merge
    with ``sharding.merge_population_state_dicts``."""

    def __init__(self, population, evaluator, interval: int = 5, fraction: float = 0.25,
                 perturb: Sequence[str] = ("lr", "ent_coef"), factors: Sequence[float] = (0.8, 1.2), seed: int = 0,
                 greedy: bool = True):
        if population.n_members != evaluator.members:
            raise ValueError("the population has %d members, the evaluator %d" % (population.n_members, evaluator.members))
        self._configure(interval, fraction, perturb, factors, seed, greedy)
        # the group each was built on (None: a single process), read from the instance's own attributes only
        if vars(population).get("group") is not vars(evaluator).get("group"):
            raise ValueError("the population and the evaluator must both be single-process or both data-parallel on the same "
                             "group")
        self.population, self.evaluator = population, evaluator
        self.history: List[dict] = []

    def _configure(self, interval, fraction, perturb, factors, seed, greedy):
        if int(interval) < 1:
            raise ValueError("interval must be >= 1")
        if not 0.0 <= float(fraction) <= 0.5:
            raise ValueError("fraction must lie in [0, 0.5]: the bottom and top sets must not overlap")
        perturb = tuple(perturb)
        for key in perturb:
            if key in ("gamma", "lam"):
                raise ValueError("%s is a discount in [0, 1] that a factor above 1 could leave: it cannot be perturbed" % key)
            if key not in PERTURBABLE:
                raise ValueError("unknown hyper-parameter %r; perturbable: %s" % (key, ", ".join(PERTURBABLE)))
        factors = tuple(float(f) for f in factors)
        if not factors or not all(math.isfinite(f) and f > 0 for f in factors):
            raise ValueError("factors must be a non-empty sequence of finite positive numbers")
        self.interval, self.fraction, self.perturb, self.factors = int(interval), float(fraction), perturb, factors
        self.seed, self.greedy = int(seed), bool(greedy)

    def step(self) -> Dict[str, torch.Tensor]:
        """One training iteration of every member (``PPOPopulation.train_iteration``'s statistics), then, when the
        iteration count reaches a multiple of ``interval``, a ready event (appended to ``history``)."""
        stats = self.population.train_iteration()
        if self.population.iteration % self.interval == 0:
            self.ready()
        return stats

    def ready(self) -> dict:
        """The ready event: evaluate, rank, exploit, explore. Returns its ``history`` entry."""
        pop, it = self.population, self.population.iteration
        results = self.evaluator.evaluate(pop.policies, greedy=self.greedy)
        fitness = torch.tensor([float(r.returns.double().mean()) for r in results], dtype=torch.float64)
        ranking = rank_members(fitness.tolist())
        bottom, top = truncation(ranking, self.fraction)
        copies = [(p, draw_source(self.seed, it, p, top)) for p in bottom]
        sources = {q: pop.member_state_dict(q) for q in sorted({q for _, q in copies})}   # taken before any member changes
        factors = {}
        for p, q in copies:
            pop.load_member_state_dict(p, sources[q])
            factors[p] = {key: draw_factor(self.seed, it, p, key, self.factors) for key in self.perturb}
            pop.set_member_hyperparameters(p, {key: pop.hyperparameters[p][key] * f for key, f in factors[p].items()})
        event = {"iteration": it, "fitness": fitness, "ranking": ranking, "copies": copies, "factors": factors,
                 "hyperparameters": copy.deepcopy(pop.hyperparameters)}
        self.history.append(event)
        return event

    def state_dict(self) -> dict:
        """The population's ``state_dict()``, this controller's settings and its history: a run resumed from it continues
        bit for bit (the evaluator keeps no state between calls)."""
        return {"population": self.population.state_dict(),
                "settings": {"interval": self.interval, "fraction": self.fraction, "perturb": self.perturb,
                             "factors": self.factors, "seed": self.seed, "greedy": self.greedy},
                "history": copy.deepcopy(self.history)}

    def load_state_dict(self, sd: dict):
        self._configure(**sd["settings"])
        self.population.load_state_dict(sd["population"])
        self.history = copy.deepcopy(sd["history"])
