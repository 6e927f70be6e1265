"""wab_gym_b200 — B200-native batched simulator for the Wolves-and-Bushes grid world.

Public surface (mirrors ``/root/reference/wab_env.py``):
  * ``default_game_options`` — same keys/values as the reference (``wab_env.py:11-39``)
  * ``WolvesAndBushesEnv``   — single-env gym-style compat class (``reset()``, ``step(a)``)
  * ``VecEnv``               — N lockstep envs on device-resident torch tensors
  * ``Evaluator``            — complete-episode evaluation of a policy, replayable episode by episode
  * ``PPOPopulation``        — P PPO policies trained side by side on one VecEnv, each bit for bit its standalone run
  * ``PopulationEvaluator``  — P policies evaluated on the same episodes in one launch per step
  * ``PopulationBasedTraining`` — exploit and explore over a ``PPOPopulation`` ranked by a ``PopulationEvaluator``

The compute path is hand-written sm_100a CUDA behind the C ABI of ``include/wab_b200.h``; there is
no CPU fallback, and importing the env classes fails loudly if the library cannot be loaded.
"""
from .config import GameConfig, default_game_options  # noqa: F401

__all__ = ["GameConfig", "default_game_options", "VecEnv", "ObsBatch", "WolvesAndBushesEnv", "Evaluator", "EvalResult", "PPOPopulation",
           "PopulationEvaluator", "PopulationBasedTraining"]


def __getattr__(name):  # lazy: `import wab_gym_b200.config` must work without torch / CUDA
    if name in ("VecEnv", "ObsBatch"):
        from . import vec_env
        return getattr(vec_env, name)
    if name in ("Evaluator", "EvalResult", "PopulationEvaluator"):
        from . import evaluate
        return getattr(evaluate, name)
    if name == "PPOPopulation":
        from .population import PPOPopulation
        return PPOPopulation
    if name == "PopulationBasedTraining":
        from .pbt import PopulationBasedTraining
        return PopulationBasedTraining
    if name == "WolvesAndBushesEnv":
        from .env import WolvesAndBushesEnv
        return WolvesAndBushesEnv
    raise AttributeError(name)
