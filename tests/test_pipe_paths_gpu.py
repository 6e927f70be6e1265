"""The pipeline kernel's rule warp (env_step_pipe) runs the common step as straight-line code and sends each rare path
through a warp-uniform test: a tie of a revealed block, the depletion log of an env that ate a bush empty, wolves, an eat
(and one that finds its cell in the log), a spawn, a reset. At configs[1]'s scale, with option sets and capacities chosen
so that every one of those paths runs — the depletion log and the wolf slots overflowing, fp64 food, no auto-reset, a
ragged last warp whose absent envs step a neutral state — every output, the hidden state and the statistics of pipeline
launches equal what single-step launches give."""
import numpy as np
import pytest
import torch

from tests.util import OPTION_SETS

pytestmark = pytest.mark.gpu

CASES = {
    # name: (n, option set, VecEnv keywords)
    "small_caps": (4096, "dense", {"log_cap": 2, "wolf_cap": 2}),
    "f64_no_auto_reset": (4096, "defaults", {"force_f64_food": True, "auto_reset": False}),
    "ragged": (4093, "defaults", {}),
    "restrict_view": (4096, "restrict_view", {}),
    "dense": (4096, "dense", {}),
    "tiny_bushes": (4093, "tiny_bushes", {"log_cap": 4}),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_pipe_rare_paths_equal_single_steps(case, monkeypatch):
    from wab_gym_b200 import VecEnv
    monkeypatch.setenv("WAB_PIPE", "2")
    n, opts, kw = CASES[case]
    overrides, _ = OPTION_SETS[opts]
    a = VecEnv(n, overrides, seed=5, features=True, **kw)
    b = VecEnv(n, overrides, seed=5, features=True, **kw)
    assert a.lanes_per_env > 1
    gen = torch.Generator(device="cuda").manual_seed(3)
    a.reset(); b.reset()
    T = 192
    for launch in range(2):
        acts = torch.randint(0, a.n_actions, (T, n), dtype=torch.uint8, device="cuda", generator=gen)
        acts[5 + launch, ::61] = 250                                     # bad actions
        assert "pipe" in a.step_kernel_name(T)
        oa, ra, da, ia = a.step_many(acts)
        for t in range(T):
            ob, rb, db, ib = b.step(acts[t])
            for x, y in zip(oa, ob):
                assert torch.equal(x[t], y), (case, launch, t)
            assert torch.equal(ra[t], rb) and torch.equal(da[t], db), (case, launch, t)
            assert torch.equal(ia["info"][t], ib["info"]) and torch.equal(ia["features"][t], ib["features"]), (case, launch, t)
        sa, sb = a.export_state(), b.export_state()
        for k in sa:
            assert np.array_equal(sa[k], sb[k]), (case, launch, k)
    st = a.stats()
    assert st == b.stats()
    assert st["eats"] > 0 and st["bad_actions"] > 0
    if kw.get("auto_reset", True):
        assert st["episodes"] > 0
    if case == "small_caps":
        assert st["overflows"] > 0
    a.close(); b.close()
