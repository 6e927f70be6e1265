"""Evaluation on the host: ``first_episodes`` against a plain Python loop, ``EvalResult.summary`` against hand-computed
values, and the evaluator's refusal of networks the tensor-core forward does not serve. No GPU needed."""
import math

import pytest
import torch
import torch.nn as nn

from wab_gym_b200.evaluate import EvalResult, Evaluator, check_policy, first_episodes
from wab_gym_b200.policy import Policy


def _loop(reward, done, info, k):
    """The first k episodes of each env, one step after another as EpisodeMonitor walks them."""
    T, N = reward.shape
    out = {key: [[None] * k for _ in range(N)] for key in ("returns", "lengths", "outcome", "eats")}
    for n in range(N):
        j, ret, length, eats = 0, 0.0, 0, 0
        for t in range(T):
            if j == k:
                break
            ret += float(reward[t, n])
            length += 1
            eats += (int(info[t, n]) >> 2) & 1
            if bool(done[t, n]):
                out["returns"][n][j], out["lengths"][n][j] = ret, length
                out["outcome"][n][j], out["eats"][n][j] = int(info[t, n]) & 3, eats
                j, ret, length, eats = j + 1, 0.0, 0, 0
    return out


def _record(T, N, p_done, seed, min_episodes=None):
    g = torch.Generator().manual_seed(seed)
    reward = (torch.randn(T, N, generator=g) * 3).float()
    done = torch.rand(T, N, generator=g) < p_done
    if min_episodes is not None:                       # guarantee enough episodes: a done every few steps at the end
        done[-2 * min_episodes::2] = True
    outcome = torch.randint(1, 4, (T, N), generator=g)
    ate = torch.randint(0, 2, (T, N), generator=g)
    noise_bits = torch.randint(0, 4, (T, N), generator=g) << 3          # bad-action and final-status bits are ignored
    info = (torch.where(done, outcome, 0) | (ate << 2) | noise_bits).to(torch.uint8)
    return reward, done, info


@pytest.mark.parametrize("T,N,p_done,k,seed", [(40, 17, 0.2, 1, 0), (60, 9, 0.3, 3, 1), (25, 31, 0.9, 2, 2),
                                               (30, 5, 0.05, 1, 3)])
def test_first_episodes_matches_a_python_loop(T, N, p_done, k, seed):
    reward, done, info = _record(T, N, p_done, seed, min_episodes=k)
    returns, lengths, outcome, eats = first_episodes(reward, done, info, k)
    assert returns.dtype == torch.float64 and lengths.dtype == torch.int32 and outcome.dtype == torch.uint8
    assert eats.dtype == torch.int32 and returns.shape == (N, k)
    want = _loop(reward, done, info, k)
    for n in range(N):
        for j in range(k):
            assert float(returns[n, j]) == want["returns"][n][j], (n, j)
            assert int(lengths[n, j]) == want["lengths"][n][j] and int(outcome[n, j]) == want["outcome"][n][j], (n, j)
            assert int(eats[n, j]) == want["eats"][n][j], (n, j)


def test_first_episodes_edge_cases():
    # env 0: exactly k = 2 episodes; env 1: more than k, the first of length 1; env 2: every step is an episode
    T = 6
    done = torch.tensor([[0, 1, 1], [0, 0, 1], [1, 1, 1], [0, 0, 1], [0, 1, 1], [1, 0, 1]], dtype=torch.bool)
    reward = torch.arange(T * 3, dtype=torch.float32).reshape(T, 3) * 0.25
    info = (torch.where(done, 2, 0) | (torch.ones(T, 3, dtype=torch.int64) << 2)).to(torch.uint8)
    info[2, 0] = 1 | 4                                 # env 0's first episode finished
    returns, lengths, outcome, eats = first_episodes(reward, done, info, 2)
    assert lengths.tolist() == [[3, 3], [1, 2], [1, 1]]
    assert outcome.tolist() == [[1, 2], [2, 2], [2, 2]]
    assert eats.tolist() == lengths.tolist()
    assert returns[1].tolist() == [float(reward[0, 1]), float(reward[1, 1]) + float(reward[2, 1])]
    assert returns[2].tolist() == [float(reward[0, 2]), float(reward[1, 2])]
    assert torch.equal(first_episodes(reward, done, info, 1)[0], returns[:, :1].contiguous())
    with pytest.raises(ValueError, match="fewer than k"):
        first_episodes(reward, done, info, 3)         # env 0 completes only two
    with pytest.raises(ValueError):
        first_episodes(reward, done[:-1], info, 1)
    with pytest.raises(ValueError):
        first_episodes(reward, done, info, 0)


def test_summary_by_hand():
    res = EvalResult(returns=torch.tensor([[1.0, 3.0], [2.0, -2.0]], dtype=torch.float64),
                     lengths=torch.tensor([[10, 20], [30, 40]], dtype=torch.int32),
                     outcome=torch.tensor([[1, 2], [3, 1]], dtype=torch.uint8),
                     eats=torch.zeros(2, 2, dtype=torch.int32), first_features=torch.zeros(2, 2, 28, dtype=torch.uint8))
    s = res.summary()
    assert s["episodes"] == 4 and s["mean_return"] == 1.0 and s["mean_length"] == 25.0
    assert s["std_return"] == pytest.approx(math.sqrt(14.0 / 4.0), rel=1e-15)   # population std of 1, 3, 2, -2
    assert (s["finished"], s["starved"], s["killed"]) == (0.5, 0.25, 0.25)


class _Wider(Policy):
    def __init__(self, obs_dim, n_actions):
        super().__init__(obs_dim, n_actions)
        self.affine2 = nn.Linear(128, 200)
        self.affine3 = nn.Linear(200, 128)


@pytest.mark.parametrize("case", ["wider_trunk", "nine_actions", "input_width", "float64", "not_a_policy"])
def test_evaluator_refuses_other_networks_before_touching_a_device(case):
    dim = 449
    pol = {"wider_trunk": lambda: _Wider(dim, 6), "nine_actions": lambda: Policy(dim, 9),
           "input_width": lambda: Policy(dim + 1, 6), "float64": lambda: Policy(dim, 6).double(),
           "not_a_policy": lambda: nn.Sequential(nn.Linear(dim, 6))}[case]()
    with pytest.raises(ValueError):
        check_policy(pol, dim)
    ev = Evaluator.__new__(Evaluator)                  # no env, no device: evaluate must refuse before it needs either
    ev.flat_dim = dim
    with pytest.raises(ValueError):
        ev.evaluate(pol)
    check_policy(Policy(dim, 6), dim)                  # the reference's network passes
    check_policy(Policy(dim, 8), dim)
