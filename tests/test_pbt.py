"""Population-based training's host side without a GPU: ranking with ties, the truncation sets, the keyed source and
factor draws (reproducible, independent of every global generator) and the controller's refusals."""
import random

import numpy as np
import pytest
import torch

from wab_gym_b200.pbt import PERTURBABLE, PopulationBasedTraining, draw_factor, draw_source, rank_members, truncation


class _Population:
    """What the controller reads at construction: the member count. Anything else is a device call it must not make."""

    def __init__(self, members):
        self.n_members = members

    def __getattr__(self, name):
        raise AssertionError("PopulationBasedTraining touched the population (%s) before refusing" % name)


class _Evaluator:
    def __init__(self, members):
        self.members = members


def test_ranking_is_highest_first_with_ties_to_the_lower_index():
    assert rank_members([1.0, 3.0, 2.0]) == [1, 2, 0]
    assert rank_members([2.0, 5.0, 2.0, 5.0, -1.0]) == [1, 3, 0, 2, 4]
    assert rank_members([0.0] * 4) == [0, 1, 2, 3]
    assert rank_members([float("-inf"), 0.0]) == [1, 0]


@pytest.mark.parametrize("P", [1, 2, 3, 4, 7, 16, 64])
@pytest.mark.parametrize("fraction", [0.0, 0.1, 0.25, 0.3, 0.5])
def test_truncation_sets(P, fraction):
    ranking = list(np.random.default_rng(P).permutation(P))
    bottom, top = truncation(ranking, fraction)
    k = int(np.floor(fraction * P))
    assert len(bottom) == len(top) == k
    assert top == ranking[:k] and bottom == (ranking[P - k:] if k else [])
    assert not set(top) & set(bottom)


def test_draws_are_keyed_and_ignore_the_global_generators():
    top = [5, 2, 9]
    first = [(draw_source(7, it, p, top), draw_factor(7, it, p, "lr", (0.8, 1.2))) for it in range(4) for p in range(8)]
    torch.manual_seed(123)
    random.seed(4)
    np.random.seed(5)
    torch.rand(100)
    again = [(draw_source(7, it, p, top), draw_factor(7, it, p, "lr", (0.8, 1.2))) for it in range(4) for p in range(8)]
    assert first == again
    assert all(q in top for q, _ in first) and all(f in (0.8, 1.2) for _, f in first)
    # the key matters: other seeds, iterations and members draw differently somewhere
    assert len({q for q, _ in first}) > 1 and len({f for _, f in first}) == 2
    assert [draw_source(8, it, p, top) for it in range(4) for p in range(8)] != [q for q, _ in first]
    # a key's factor does not depend on which other keys are perturbed, and different keys draw independently
    lr = [draw_factor(7, 3, p, "lr", (0.5, 1.0, 2.0)) for p in range(32)]
    ent = [draw_factor(7, 3, p, "ent_coef", (0.5, 1.0, 2.0)) for p in range(32)]
    assert lr != ent


def test_factor_draws_cover_every_perturbable_key():
    for key in PERTURBABLE:
        assert draw_factor(0, 1, 2, key, (3.0,)) == 3.0
    with pytest.raises(ValueError):
        draw_factor(0, 1, 2, "gamma", (3.0,))


@pytest.mark.parametrize("kwargs, match", [
    (dict(perturb=("gamma",)), "gamma"),
    (dict(perturb=("lr", "lam")), "lam"),
    (dict(perturb=("learning_rate",)), "unknown"),
    (dict(fraction=-0.1), r"\[0, 0.5\]"),
    (dict(fraction=0.6), r"\[0, 0.5\]"),
    (dict(interval=0), "interval"),
    (dict(factors=()), "factors"),
    (dict(factors=(0.8, -1.0)), "factors"),
    (dict(factors=(float("nan"),)), "factors"),
])
def test_refusals(kwargs, match):
    with pytest.raises(ValueError, match=match):
        PopulationBasedTraining(_Population(4), _Evaluator(4), **kwargs)


def test_member_count_mismatch_is_refused():
    with pytest.raises(ValueError, match="members"):
        PopulationBasedTraining(_Population(4), _Evaluator(3))


def test_settings_are_kept():
    pbt = PopulationBasedTraining(_Population(4), _Evaluator(4), interval=3, fraction=0.5, perturb=["clip_eps"],
                                  factors=[0.5, 2], seed=9, greedy=False)
    assert (pbt.interval, pbt.fraction, pbt.perturb, pbt.factors, pbt.seed, pbt.greedy) == (3, 0.5, ("clip_eps",), (0.5, 2.0),
                                                                                           9, False)
    assert pbt.history == []
