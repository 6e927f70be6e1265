"""PPOPopulation's host side without a GPU: hyper-parameter validation and the refusals raised before any device work,
the member-local to global row translation, and GAE with per-column discounts against ``gae`` run per member."""
import pytest
import torch

from wab_gym_b200.population import HYPERPARAMETERS, PPOPopulation, member_hyperparameters, member_rows
from wab_gym_b200.ppo import PPOTrainer, gae


class _Env:
    """What the constructor reads before it touches a device: an env that raises on any other use."""

    def __init__(self, num_envs, with_features=True):
        self.num_envs, self.with_features, self.flat_dim, self.n_actions = num_envs, with_features, 449, 5

    @property
    def device(self):
        raise AssertionError("PPOPopulation touched the device before refusing")


def test_defaults_are_ppo_trainers():
    import inspect
    sig = inspect.signature(PPOTrainer.__init__).parameters
    assert HYPERPARAMETERS == {k: sig[k].default for k in HYPERPARAMETERS}
    full = member_hyperparameters([{}, {"lr": 1e-3, "gamma": 0.9}], 2)
    assert full[0] == HYPERPARAMETERS and full[1]["lr"] == 1e-3 and full[1]["gamma"] == 0.9
    assert full[1]["lam"] == HYPERPARAMETERS["lam"]
    assert member_hyperparameters(None, 3) == [HYPERPARAMETERS] * 3


@pytest.mark.parametrize("hps, match", [
    ([{"learning_rate": 1e-3}], "unknown"),
    ([{}, {}], "one dict per member"),
    ([{"clip_eps": 0.0}], "clip_eps"),
    ([{"max_grad_norm": -1.0}], "max_grad_norm"),
])
def test_hyperparameters_refused(hps, match):
    with pytest.raises(ValueError, match=match):
        member_hyperparameters(hps, 1)


@pytest.mark.parametrize("kwargs, match", [
    (dict(members=3, group=object()), "group"),
    (dict(members=0), "1 to 64"),
    (dict(members=65), "1 to 64"),
    (dict(members=3, n_envs=3 * 100), "multiple of 128"),
    (dict(members=2, n_envs=3 * 128), "multiple of 128"),
    (dict(members=2, features=False), "features"),
    (dict(members=2, epochs=0), "epochs"),
    (dict(members=2, minibatches=0), "minibatches"),
    (dict(members=2, horizon=1, minibatches=129), "minibatches"),
    (dict(members=2, hyperparameters=[{}, {"gamm": 0.9}]), "unknown"),
    (dict(members=2, hyperparameters=[{}, {"max_grad_norm": 0.0}]), "max_grad_norm"),
    (dict(members=2, policies=[None]), "one Policy per member"),
])
def test_refusals_come_before_the_device(kwargs, match):
    n_envs = kwargs.pop("n_envs", 2 * 128 if kwargs.get("members", 2) != 3 else 3 * 128)
    env = _Env(n_envs, kwargs.pop("features", True))
    with pytest.raises(ValueError, match=match):
        PPOPopulation(env, **kwargs)


def test_refuses_a_network_the_kernels_do_not_serve():
    from wab_gym_b200.policy import Policy
    env = _Env(2 * 128)
    bad = Policy(449, 5)
    bad.affine2 = torch.nn.Linear(128, 64)
    with pytest.raises(ValueError, match="reference's network"):
        PPOPopulation(env, 2, policies=[Policy(449, 5), bad])
    with pytest.raises(ValueError, match="fp32"):
        PPOPopulation(env, 2, policies=[Policy(449, 5), Policy(449, 5).double()])


@pytest.mark.parametrize("P, n, T", [(1, 128, 3), (3, 256, 5), (4, 128, 2)])
def test_member_rows_translate_local_to_global(P, n, T):
    g = torch.Generator().manual_seed(P * 1000 + n)
    perm = torch.randperm(T * n, generator=g).to(torch.int32)[: T * n // 2 + 1]
    got = member_rows(perm, P, n)
    N = P * n
    want = [[(int(i) // n) * N + p * n + int(i) % n for i in perm] for p in range(P)]
    assert got.dtype == torch.int32 and got.tolist() == want
    wide = torch.full((P, perm.numel() + 7), -1, dtype=torch.int32)
    member_rows(perm, P, n, out=wide[:, :perm.numel()])
    assert wide[:, :perm.numel()].tolist() == want and bool((wide[:, perm.numel():] == -1).all())


def test_per_column_gae_is_gae_per_member_bit_for_bit():
    P, n, T = 3, 128, 17
    gammas, lams = [0.99, 0.9, 0.999], [0.95, 0.8, 0.97]
    g = torch.Generator().manual_seed(7)
    rewards = torch.randn(T, P * n, generator=g)
    values = torch.randn(T, P * n, generator=g)
    dones = torch.rand(T, P * n, generator=g) < 0.1
    boot = torch.randn(P * n, generator=g)
    gamma = torch.tensor(gammas, dtype=torch.float32).repeat_interleave(n)
    gamma_lam = torch.tensor([a * b for a, b in zip(gammas, lams)], dtype=torch.float32).repeat_interleave(n)
    adv, ret = gae(rewards, dones, values, boot, gamma, None, gamma_lam=gamma_lam)
    for p in range(P):
        sl = slice(p * n, (p + 1) * n)
        a, r = gae(rewards[:, sl].contiguous(), dones[:, sl].contiguous(), values[:, sl].contiguous(), boot[sl].contiguous(),
                   gammas[p], lams[p])
        assert torch.equal(adv[:, sl], a) and torch.equal(ret[:, sl], r)
