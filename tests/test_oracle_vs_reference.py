"""Live differential test: C oracle vs the unmodified reference run under oracle/ref_shim.
The live comparisons run only where the reference sources are present (WAB_REFERENCE_DIR); tests/golden carries the
reference's behaviour everywhere else."""
import importlib.util
import os
import sys
import types

import numpy as np
import pytest

from oracle import ref_shim
from oracle.wab_oracle import OracleEnv
from tests.util import OPTION_SETS, pick_action

needs_reference = pytest.mark.skipif(not ref_shim.reference_available(), reason="reference sources not present")


@pytest.mark.reference
@needs_reference
@pytest.mark.parametrize("name", ["defaults", "six_actions_random_start", "dense", "tiny_bushes"])
def test_oracle_matches_reference_live(name):
    overrides, greedy = OPTION_SETS[name]
    seed, env_id, n_steps = 17, 3, 120
    ref = ref_shim.make_env(overrides, seed=seed, env_id=env_id)
    orc = OracleEnv(overrides, seed=seed, env_id=env_id)
    o_obs = orc.reset()
    r_obs = ref._get_obs()
    rng = np.random.default_rng(5)

    def check(tag):
        for p in range(3):
            assert np.array_equal(np.asarray(r_obs[p]).astype(np.uint8), o_obs[0][p]), (tag, p)
        assert (int(r_obs[3]), int(r_obs[4]), int(r_obs[5])) == o_obs[1:], tag
        hr, ho = ref_shim.hidden_state(ref), orc.hidden_state()
        for k in ("x", "y", "food", "role", "status", "turn", "wolves", "bushes"):
            assert hr[k] == ho[k], (tag, k)

    check("init")
    done = False
    for n in range(n_steps):
        if done:
            r_obs, o_obs = ref.reset(), orc.reset()
            check(("reset", n))
        a = pick_action(rng, o_obs[0], orc.n_actions, greedy)
        r_obs, rr, done, _ = ref.step(a)
        o_obs, orr, od = orc.step(a)
        assert float(rr) == orr and bool(done) == od, (n, rr, orr)
        check(("step", n, a))


def test_clip_write_through_caps_food_at_one():
    """SURVEY §7 step 1: eating at full food must give observation food 39 (not 44) and reward 0.1 — what the reference
    returns, checked against the reference itself where its sources are present."""
    for env_id in range(200):
        orc = OracleEnv(None, seed=99, env_id=env_id)
        if orc.reset()[0][1][5, 5] == 1:
            break
    else:
        pytest.skip("no env starts on a bush")
    obs, reward, done = orc.step(4)
    assert obs[1] == 39 and abs(reward - 0.1) < 1e-12
    if ref_shim.reference_available():
        ref = ref_shim.make_env(None, seed=99, env_id=env_id)
        obs, reward, done, _ = ref.step(4)
        assert obs[3] == 39 and abs(reward - 0.1) < 1e-12


@pytest.mark.reference
@needs_reference
def test_reference_unit_tests_pass_under_shim():
    """The reference's own known-answer tests (wab_env_test.py: PragmaticObsWrapper) run unmodified."""
    import unittest
    mod = ref_shim.load_reference()
    sys.modules["wab_env"] = mod
    try:
        path = os.path.join(ref_shim.REFERENCE_DIR, "wab_env_test.py")
        spec = importlib.util.spec_from_file_location("wab_env_test_reference", path)
        tmod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(tmod)
        suite = unittest.defaultTestLoader.loadTestsFromModule(tmod)
        result = unittest.TextTestRunner(verbosity=0).run(suite)
        assert result.testsRun == 3 and result.wasSuccessful()
    finally:
        sys.modules.pop("wab_env", None)
