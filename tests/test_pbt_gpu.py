"""Population-based training on the B200: with fraction 0 it is the plain population bit for bit; a ready event copies
policy, Adam state and hyper-parameters from the drawn source and scales them by the recorded factors; members that
were not copied go on as in the plain population; and a run resumed from ``state_dict()`` ends bit-identical."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu

P, n, T = 4, 128, 8
HPS = [{"lr": 3e-4 * (1 + p), "ent_coef": 0.01 * (p + 1)} for p in range(P)]


def _policies():
    from wab_gym_b200.policy import Policy
    torch.manual_seed(21)
    return [Policy(449, 5) for _ in range(P)]


def _population(policies):
    from wab_gym_b200 import PPOPopulation, VecEnv
    env = VecEnv(P * n, seed=6, features=True)
    return PPOPopulation(env, P, hyperparameters=copy.deepcopy(HPS), policies=[copy.deepcopy(p) for p in policies],
                         horizon=T, epochs=2, minibatches=2)


def _pbt(policies, **kw):
    from wab_gym_b200 import PopulationBasedTraining, PopulationEvaluator
    return PopulationBasedTraining(_population(policies), PopulationEvaluator(P, n, seed=2), **kw)


def _same_member(pa, p, pb, q):
    """Member p of population pa and member q of pb hold the same weights, Adam state and hyper-parameters."""
    if not all(torch.equal(a, b) for a, b in zip(pa.policies[p].parameters(), pb.policies[q].parameters())):
        return False
    sa, sb = pa.optimizers[p].state_dict(), pb.optimizers[q].state_dict()
    for i in sa["state"]:
        if sa["state"][i]["step"] != sb["state"][i]["step"]:
            return False
        if not all(torch.equal(sa["state"][i][k], sb["state"][i][k]) for k in ("exp_avg", "exp_avg_sq")):
            return False
    return (pa.hyperparameters[p] == pb.hyperparameters[q]
            and sa["param_groups"][0]["lr"] == sb["param_groups"][0]["lr"] == pa.hyperparameters[p]["lr"])


def test_fraction_zero_is_the_plain_population():
    pols = _policies()
    plain = _population(pols)
    pbt = _pbt(pols, interval=1, fraction=0.0)
    for _ in range(3):
        plain.train_iteration()
        pbt.step()
    assert len(pbt.history) == 3 and all(e["copies"] == [] for e in pbt.history)
    for p in range(P):
        assert _same_member(plain, p, pbt.population, p)
    assert pbt.history[-1]["fitness"].dtype == torch.float64 and pbt.history[-1]["fitness"].shape == (P,)


def test_ready_event_copies_and_perturbs():
    pols = _policies()
    plain = _population(pols)
    pbt = _pbt(pols, interval=2, fraction=0.5, perturb=("lr", "ent_coef", "clip_eps"), factors=(0.5, 2.0), seed=3)
    pop = pbt.population
    pbt.step()
    plain.train_iteration()
    plain.train_iteration()
    pop.train_iteration()                                  # iteration 2 by hand, so the state before the event is known
    before = [pop.member_state_dict(q) for q in range(P)]
    event = pbt.ready()
    assert event["iteration"] == 2 and len(event["copies"]) == 2
    from wab_gym_b200.pbt import rank_members
    ranking = event["ranking"]
    assert ranking == rank_members(event["fitness"].tolist())
    top, bottom = ranking[:2], ranking[2:]
    copied = {p for p, _ in event["copies"]}
    assert copied == set(bottom) and all(q in top for _, q in event["copies"])
    for p, q in event["copies"]:
        src = before[q]
        assert all(torch.equal(a.cpu(), src["policy"][k]) for k, a in pop.policies[p].state_dict().items())
        osd = pop.optimizers[p].state_dict()
        for i, st in src["optimizer"]["state"].items():
            assert all(torch.equal(osd["state"][i][k], st[k]) for k in ("exp_avg", "exp_avg_sq"))
        f = event["factors"][p]
        assert set(f) == {"lr", "ent_coef", "clip_eps"} and all(v in (0.5, 2.0) for v in f.values())
        for key, hp in pop.hyperparameters[p].items():
            assert hp == (src["hyperparameters"][key] * f[key] if key in f else src["hyperparameters"][key])
        assert osd["param_groups"][0]["lr"] == pop.hyperparameters[p]["lr"]
        assert event["hyperparameters"][p] == pop.hyperparameters[p]
    # the members that were not copied are untouched, and go on exactly as in the plain population
    for q in top:
        assert _same_member(plain, q, pop, q)
    plain.train_iteration()
    pbt.step()
    for q in top:
        assert _same_member(plain, q, pop, q)


@pytest.mark.parametrize("split", [1, 2])
def test_resume_is_bit_identical(split):
    pols = _policies()
    kw = dict(interval=2, fraction=0.25, perturb=("lr", "max_grad_norm", "vf_coef"), seed=5)
    whole = _pbt(pols, **kw)
    for _ in range(4):
        whole.step()
    first = _pbt(pols, **kw)
    for _ in range(split):
        first.step()
    sd = first.state_dict()
    resumed = _pbt(_policies(), interval=9, fraction=0.0)   # other settings: load_state_dict restores them
    resumed.load_state_dict(sd)
    assert resumed.interval == 2 and resumed.fraction == 0.25 and resumed.seed == 5
    for _ in range(4 - split):
        resumed.step()
    assert len(resumed.history) == len(whole.history) == 2
    for a, b in zip(resumed.history, whole.history):
        assert a["copies"] == b["copies"] and a["factors"] == b["factors"] and torch.equal(a["fitness"], b["fitness"])
        assert a["hyperparameters"] == b["hyperparameters"] and a["ranking"] == b["ranking"]
    for p in range(P):
        assert _same_member(whole.population, p, resumed.population, p)
