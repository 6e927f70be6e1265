"""``WolvesAndBushesEnv`` — the reference's single-environment gym surface on the CUDA path.

Drop-in for ``/root/reference/wab_env.py:103-342``: same constructor arguments, ``reset()`` returning
the 7-tuple ``(wolf_grid, bush_grid, ostrich_grid, food, role, alive_starved_killed, view_mask)``
(``wab_env.py:374-385``; the first six are the tuple the Readme documents), ``step(action)`` returning
``(obs, reward, done, {})``, ``action_space`` / ``observation_space`` / ``spec`` / ``metadata`` /
``game_options`` attributes, no auto-reset (stepping after ``done`` keeps returning ``done``,
``wab_env.py:328-340``) and float64 food arithmetic. It is a batch of one on the same kernels as
``VecEnv`` (through the host-buffer C-ABI calls); it exists for API parity and differential tests,
not for throughput.

Differences that are deliberate: randomness comes from keyed Philox draws (``seed``, ``env_id``)
instead of the global ``np.random`` stream (the reference has no seeding: ``# TODO random seed``,
``wab_env.py:233``).
"""
from __future__ import annotations

import ctypes
from typing import Optional

import numpy as np

from . import _lib
from .config import GATHERER_TILE_MASK, LOOKOUT_TILE_MASK, GameConfig, default_game_options


class Discrete:
    """Stand-in for ``gym.spaces.Discrete`` (gym is not a dependency)."""

    def __init__(self, n):
        self.n = int(n)
        self.shape = ()
        self.dtype = np.int64
        self._rng = np.random.default_rng()

    def sample(self):
        return int(self._rng.integers(self.n))

    def contains(self, x):
        return 0 <= int(x) < self.n

    def __repr__(self):
        return "Discrete(%d)" % self.n


class Box:
    def __init__(self, low, high, shape, dtype=int):
        self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), dtype

    def __repr__(self):
        return "Box(%r, %r, %r)" % (self.low, self.high, self.shape)


class Tuple:
    def __init__(self, spaces):
        self.spaces = tuple(spaces)

    def __getitem__(self, i):
        return self.spaces[i]

    def __len__(self):
        return len(self.spaces)

    def __repr__(self):
        return "Tuple(%s)" % ", ".join(map(repr, self.spaces))


class EnvSpec:
    """Same fields as the reference's ``DummySpec`` (wab_env.py:87-100)."""

    def __init__(self, id, reward_threshold=None, nondeterministic=False, max_episode_steps=None):
        self.id = id
        self.reward_threshold = reward_threshold
        self.nondeterministic = nondeterministic
        self.max_episode_steps = max_episode_steps


def _hptr(a: np.ndarray):
    return ctypes.c_void_p(a.ctypes.data)


class WolvesAndBushesEnv:
    metadata = {"render.modes": ["rgb_array"], "video.frames_per_second": 12}  # wab_env.py:104

    def __init__(self, game_options=default_game_options, render=False, *, seed: int = 0, env_id: int = 0,
                 device: int = 0):
        self._h = None
        self.game_options = game_options  # held by reference, like wab_env.py:107
        for key in ("width", "height", "max_turns", "gatherer_only", "lookout_only"):
            game_options[key]  # KeyError on missing options, as the reference's dict lookups
        self._game = GameConfig.from_options(game_options, auto_reset=False, force_f64_food=True, wolf_cap=64)
        self.lookout_tile_mask = LOOKOUT_TILE_MASK.astype(np.int64)    # wab_env.py:109-123
        self.gatherer_tile_mask = GATHERER_TILE_MASK.astype(np.int64)  # wab_env.py:125-139
        self.spec = EnvSpec(id="WolvesAndBushes-v0", max_episode_steps=game_options["max_turns"],
                            reward_threshold=80)                       # wab_env.py:140-146
        self.action_space = Discrete(self._game.n_actions)             # wab_env.py:188-191
        w, h = game_options["width"], game_options["height"]
        self.observation_space = Tuple((                               # wab_env.py:193-229
            Box(0, 1, (w, h), int), Box(0, 1, (w, h), int), Box(0, 1, (w, h), int),
            Discrete(game_options["turns_to_empty_food"] + 1), Discrete(2), Discrete(3)))
        self._lib = _lib.load()
        self._seed, self._env_id, self._device = int(seed), int(env_id), int(device)
        cs = self._game.to_struct()
        thr = np.ascontiguousarray(self._game.bush_thr, dtype=np.uint32)
        handle = ctypes.c_void_p()
        _lib.check(self._lib.wab_vec_create(ctypes.byref(cs), thr.ctypes.data, len(thr), 1,
                                            int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_id), int(device),
                                            ctypes.byref(handle)))
        self._h = handle
        self._grids = np.zeros((3, w, h), dtype=np.uint8)
        self._b = {k: np.zeros(1, dtype=np.uint8) for k in ("action", "food", "role", "status", "done", "info")}
        self._reward = np.zeros(1, dtype=np.float32)
        self.current_turn = 0
        self.reset()                                                   # wab_env.py:186

    # ------------------------------------------------------------------ gym surface
    def reset(self):
        _lib.check(self._lib.wab_vec_reset_host(self._h, _hptr(self._grids), _hptr(self._b["food"]),
                                                _hptr(self._b["role"]), _hptr(self._b["status"]), None))
        self.current_turn = 0
        return self._get_obs()

    def step(self, actions):
        n = self._game.n_actions
        a = int(actions)
        if not -n <= a < n:  # DataFrame.iloc semantics at wab_env.py:253 (negative indices wrap)
            raise IndexError("single positional indexer is out-of-bounds")
        self._b["action"][0] = a % n
        b = self._b
        _lib.check(self._lib.wab_vec_step_host(self._h, _hptr(b["action"]), _hptr(self._grids), _hptr(b["food"]),
                                               _hptr(b["role"]), _hptr(b["status"]), _hptr(self._reward),
                                               _hptr(b["done"]), _hptr(b["info"]), None))
        self.current_turn += 1
        info = int(b["info"][0])
        o = self.game_options
        reward = 0                                                     # wab_env.py:251
        if (info >> 2) & 1:
            reward += o["reward_for_eating"]                           # wab_env.py:313
        reward += (o["reward_per_turn"], o["reward_for_finishing"], o["reward_for_starving"],
                   o["reward_for_being_killed"])[info & 3]             # wab_env.py:328-340
        return self._get_obs(), reward, bool(b["done"][0]), {}

    def _get_obs(self):
        role = int(self._b["role"][0])
        if self.game_options["restrict_view"]:                         # wab_env.py:361-368
            view_mask = self.gatherer_tile_mask if role == 1 else self.lookout_tile_mask
        else:
            view_mask = np.zeros((11, 11))
        g = self._grids.astype(np.float64)                             # reference grids are float64 zeros/ones
        return (g[0], g[1], g[2], int(self._b["food"][0]), role, int(self._b["status"][0]), view_mask)

    def render(self, mode="rgb_array", scale=32, draw_health=True):
        """RGB frame in the reference's colours (wab_env.py:468-502): wolves red, bushes green, ostriches blue."""
        wolves, bushes, ostriches = (self._grids[p].astype(np.uint8) for p in range(3))
        status = int(self._b["status"][0])
        image = np.zeros(self._grids.shape[1:] + (3,), dtype=np.uint8)
        image[:, :, 0], image[:, :, 1], image[:, :, 2] = 255 * wolves, 255 * bushes, 255 * ostriches
        empty = (image[:, :, 0] == 0) & (image[:, :, 1] == 0) & (image[:, :, 2] == 0)
        image[empty] = 127 if status == 2 else 255
        if status != 2 and self.game_options["restrict_view"]:
            mask = self.gatherer_tile_mask if int(self._b["role"][0]) == 1 else self.lookout_tile_mask
            image[mask == 1] = 0
        image = image.repeat(scale, axis=0).repeat(scale, axis=1)
        if draw_health:
            try:
                from PIL import Image, ImageDraw
                im = Image.fromarray(image)
                ImageDraw.Draw(im).text((0, 0), str(int(self._b["food"][0])), fill="blue")
                return np.array(im)
            except ImportError:
                pass
        return image

    # ------------------------------------------------------------------ copy.deepcopy / pickle
    def __getstate__(self):
        """Options, keys, the env's state record (wab_vec_save_state) and the last observation: ``copy.deepcopy(env)`` and
        ``pickle`` give an env that continues exactly like this one under the same actions."""
        import torch
        dev = torch.device("cuda", self._device)
        buf = torch.empty(int(self._lib.wab_vec_state_record_bytes(self._h)), dtype=torch.uint8, device=dev)
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)     # the copy below reads buf on this stream
        _lib.check(self._lib.wab_vec_save_state(self._h, None, 1, ctypes.c_void_p(buf.data_ptr()), stream))
        return {"game_options": self.game_options, "seed": self._seed, "env_id": self._env_id, "device": self._device,
                "record": buf.cpu().numpy(), "grids": self._grids.copy(), "b": {k: v.copy() for k, v in self._b.items()},
                "reward": self._reward.copy(), "current_turn": self.current_turn}

    def __setstate__(self, state):
        import torch
        self.__init__(state["game_options"], seed=state["seed"], env_id=state["env_id"], device=state["device"])
        dev = torch.device("cuda", self._device)
        rec = torch.from_numpy(np.ascontiguousarray(state["record"], dtype=np.uint8)).to(dev)
        rejected = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(self._lib.wab_vec_load_state(self._h, ctypes.c_void_p(rec.data_ptr()), None, 1, _lib.WabObs(0, 0, 0, 0),
                                                ctypes.c_void_p(rejected.data_ptr()),
                                                ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        if int(rejected.item()):
            raise ValueError("the pickled env state does not fit these options")
        self._grids[...] = state["grids"]
        for k, v in state["b"].items():
            self._b[k][...] = v
        self._reward[...] = state["reward"]
        self.current_turn = state["current_turn"]

    def seed(self, seed=None):
        return []

    def close(self):
        if getattr(self, "_h", None):
            self._lib.wab_vec_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
