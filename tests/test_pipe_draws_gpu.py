"""The two-warp pipeline's rule warp makes each step's keyed draws (this lane's slide blocks and the spawn draw) before
the rules and hands them in (step_draws, env_step with DRAWN). At configs[1]'s size, long enough that resets, bad
actions, wolves and eaten-empty bushes all occur, every output equals what single-step launches give. (Ties of a block's
high half-word with the threshold's come at 2^-15 per block: some hundreds among the 4,096 x 512 x 6 block draws.)"""
import numpy as np
import pytest
import torch

from tests.util import OPTION_SETS

pytestmark = pytest.mark.gpu


def _vec(*a, **k):
    from wab_gym_b200 import VecEnv
    return VecEnv(*a, **k)


@pytest.mark.parametrize("n", [4096, 4059])
@pytest.mark.parametrize("name", ["dense", "tiny_bushes"])
def test_drawn_steps_equal_single_steps_at_scale(n, name, monkeypatch):
    monkeypatch.setenv("WAB_PIPE", "2")
    overrides, _ = OPTION_SETS[name]
    a = _vec(n, overrides, seed=77, features=True)
    b = _vec(n, overrides, seed=77, features=True)
    assert a.lanes_per_env > 1
    gen = torch.Generator(device="cuda").manual_seed(9)
    a.reset(); b.reset()
    T = 256
    for launch in range(2):
        acts = torch.randint(0, a.n_actions, (T, n), dtype=torch.uint8, device="cuda", generator=gen)
        acts[17 + launch, ::97] = 200                                    # bad actions
        assert "pipe" in a.step_kernel_name(T)
        oa, ra, da, ia = a.step_many(acts)
        for t in range(T):
            ob, rb, db, ib = b.step(acts[t])
            for x, y in zip(oa, ob):
                assert torch.equal(x[t], y), (name, n, launch, t)
            assert torch.equal(ra[t], rb) and torch.equal(da[t], db), (name, n, launch, t)
            assert torch.equal(ia["info"][t], ib["info"]) and torch.equal(ia["features"][t], ib["features"]), (name, n, launch, t)
        sa, sb = a.export_state(), b.export_state()
        for k in sa:
            assert np.array_equal(sa[k], sb[k]), (name, n, launch, k)
    st = a.stats()
    assert st == b.stats()
    assert st["episodes"] > n and st["bad_actions"] > 0
    a.close(); b.close()
