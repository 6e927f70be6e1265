"""``VecWorld2`` — N lockstep Environment-2.0 worlds on one B200.

Batched counterpart of the reference's ``WAB_Environment2`` ("/root/reference/Environment 2.0/WAB_Environment2.py":53-134)
over ``World`` (``World.py:135-377``): a toroidal W x H world of ostriches, wolves and bushes per environment, every
entity acting once per world turn in id order (ostriches, wolves, bushes). ``turn(actions)`` performs, for every
entity i in that order, what the reference driver loop does (``Env2Tests.py:46-88``): ``get_obs(i)`` then
``take_action(i, a_i)``. The reference's bugs are kept (SURVEY Appendix C).
"""
from __future__ import annotations

import ctypes
import hashlib
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib

#: the v2 ``default_game_options`` entries the world turn reads (WAB_Environment2.py:9-50)
default_game_options_v2: Dict[str, object] = {
    "starting_role": 1, "food_per_bush": 20, "food_given_per_turn": 5, "ostrich_starting_food": 40.0,
    "lookout_view_radius": 9, "gatherer_view_radius": 5, "wolf_starting_food": 20, "wolf_food_for_eating_ostrich": 10,
    "wolf_view_radius": 6,
}


class Wab2ConfigStruct(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "abi_version", "width", "height", "n_ostriches", "n_wolves", "n_bushes", "lookout_view_radius",
        "gatherer_view_radius", "wolf_view_radius", "window_radius", "starting_role", "ostrich_starting_food",
        "wolf_starting_food", "wolf_food_for_eating_ostrich", "food_per_bush", "food_given_per_turn")]


def make_config2(width, height, n_ostriches, n_wolves, n_bushes, game_options=None, window_radius=None) -> Wab2ConfigStruct:
    o = dict(default_game_options_v2)
    if game_options:
        o.update({k: v for k, v in game_options.items() if k in o})
    for k in ("ostrich_starting_food", "wolf_starting_food", "wolf_food_for_eating_ostrich", "food_per_bush", "food_given_per_turn"):
        if float(o[k]) != int(o[k]):
            raise NotImplementedError("%s must be integer-valued on the device path" % k)
    if o["starting_role"] is None:
        raise NotImplementedError("starting_role=None is not supported on the device path")
    radius = max(int(o["lookout_view_radius"]), int(o["gatherer_view_radius"]), int(o["wolf_view_radius"]))
    return Wab2ConfigStruct(1, width, height, n_ostriches, n_wolves, n_bushes, int(o["lookout_view_radius"]),
                            int(o["gatherer_view_radius"]), int(o["wolf_view_radius"]),
                            radius if window_radius is None else int(window_radius), int(o["starting_role"]),
                            int(o["ostrich_starting_food"]), int(o["wolf_starting_food"]),
                            int(o["wolf_food_for_eating_ostrich"]), int(o["food_per_bush"]), int(o["food_given_per_turn"]))


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


class VecWorld2:
    def __init__(self, num_envs: int, width: int, height: int, n_ostriches: int, n_wolves: int, n_bushes: int,
                 game_options: Optional[dict] = None, device="cuda", seed: int = 0, env_id_base: int = 0,
                 window_radius: Optional[int] = None, observations: bool = True):
        self._h = None
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.cfg = make_config2(width, height, n_ostriches, n_wolves, n_bushes, game_options, window_radius)
        self.num_envs, self.n_entities = int(num_envs), n_ostriches + n_wolves + n_bushes
        self.n_acting = n_ostriches + n_wolves
        self.R = self.cfg.window_radius
        self.seed, self.env_id_base = int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_id_base)
        h = ctypes.c_void_p()
        _lib.check(self.lib.wab2_create(ctypes.byref(self.cfg), self.num_envs, int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_id_base),
                                        self.device.index, ctypes.byref(h)))
        self._h = h
        n, a, s = self.num_envs, self.n_acting, 2 * self.R + 1
        # storage in the handle's layout: entity-major [A, N, ...] (thread per world: the worlds of a warp are contiguous for
        # every acting entity) or world-major [N, A, ...] (warp per world: a world's windows are one run). What turn()
        # returns is always indexed [entity, world, ...] — a transposed view of the storage in the second case.
        self.world_major = bool(self.lib.wab2_output_layout(self._h))
        lead = (n, a) if self.world_major else (a, n)
        self.planes_store = torch.empty(lead + (3, s, s), dtype=torch.uint8, device=self.device) if observations else None
        self.internal_store = torch.empty(lead + (5,), dtype=torch.int32, device=self.device) if observations else None
        self.reward_store = torch.empty(lead, dtype=torch.float32, device=self.device)
        self.done_store = torch.empty(lead, dtype=torch.uint8, device=self.device)

    def _view(self, t):
        return None if t is None else (t.transpose(0, 1) if self.world_major else t)

    @property
    def planes(self):
        return self._view(self.planes_store)

    @property
    def internal(self):
        return self._view(self.internal_store)

    @property
    def reward(self):
        return self._view(self.reward_store)

    @property
    def done(self):
        return self._view(self.done_store)

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset_environment(self):
        """reset_environment() of the reference (WAB_Environment2.py:113-118) for every world."""
        _lib.check(self.lib.wab2_reset(self._h, self._stream()))

    def turn(self, actions: torch.Tensor):
        """One world turn. ``actions`` u8[A, N], A = n_ostriches + n_wolves (ostrich 0-5, wolf 0-4; bushes always act
        with 0). Returns (planes u8[A, N, 3, 2R+1, 2R+1], internal i32[A, N, 5], reward f32[A, N], done bool[A, N]),
        indexed [entity, world] (views of ``*_store``, which is world-major for the warp-per-world kernel); the
        observation of entity i is what ``get_obs(i)`` returns right before it acts (World.py:360-377)."""
        if tuple(actions.shape) != (self.n_acting, self.num_envs):
            raise ValueError("actions must have shape (n_ostriches + n_wolves, num_envs)")
        a = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.lib.wab2_turn(self._h, _ptr(a), _ptr(self.planes_store), _ptr(self.internal_store),
                                      _ptr(self.reward_store), _ptr(self.done_store), self._stream()))
        return self.planes, self.internal, self.reward, self._view(self.done_store.view(torch.bool))

    def kernel_name(self) -> str:
        return "wab2_grid_turn_kernel (warp per world)" if self.lib.wab2_kernel_kind(self._h) else "wab2_turn_kernel (thread per world)"

    def export_state(self, episode: Optional[np.ndarray] = None):
        """(state9 i32[N, E, 9], turn i32[N]); ``episode`` (i32[N], optional) receives each world's episode counter."""
        out = np.zeros((self.num_envs, self.n_entities, 9), dtype=np.int32)
        turn = np.zeros(self.num_envs, dtype=np.int32)
        ep = None if episode is None else episode.ctypes.data
        _lib.check(self.lib.wab2_export_state(self._h, out.ctypes.data, turn.ctypes.data, ep, self._stream()))
        return out, turn

    def import_state(self, state9: np.ndarray, turn: Optional[np.ndarray] = None, episode: Optional[np.ndarray] = None):
        """Inverse of ``export_state`` (tests, checkpoints): ``state9`` i32[N, E, 9] = type, x, y, table X, table Y, Visible,
        food, role, status; ``turn`` and ``episode`` i32[N] or None (unchanged)."""
        st = np.ascontiguousarray(state9, dtype=np.int32)
        if st.shape != (self.num_envs, self.n_entities, 9):
            raise ValueError("state9 must have shape (num_envs, n_entities, 9)")
        tn = None if turn is None else np.ascontiguousarray(turn, dtype=np.int32)
        ep = None if episode is None else np.ascontiguousarray(episode, dtype=np.int32)
        _lib.check(self.lib.wab2_import_state(self._h, st.ctypes.data, None if tn is None else tn.ctypes.data,
                                              None if ep is None else ep.ctypes.data, self._stream()))

    @property
    def fingerprint(self) -> int:
        """64-bit hash of the configuration fields and the seed: a checkpoint loads only into a matching handle."""
        fields = [getattr(self.cfg, name) for name, _ in Wab2ConfigStruct._fields_] + [self.seed]
        digest = hashlib.blake2b(np.asarray(fields, dtype=np.int64).tobytes(), digest_size=8).digest()
        return int.from_bytes(digest, "little")

    def state_dict(self) -> dict:
        """Every world's state on the host (synchronises): one int32 record per world = turn, episode, then the
        ``export_state`` rows; same dict shape as ``VecEnv.state_dict`` (``sharding.merge_state_dicts`` applies)."""
        episode = np.zeros(self.num_envs, dtype=np.int32)
        st, turn = self.export_state(episode)
        records = np.concatenate([turn[:, None], episode[:, None], st.reshape(self.num_envs, -1)], axis=1)
        return {"format": 1, "fingerprint": self.fingerprint, "records": torch.from_numpy(records),
                "env_ids": torch.arange(self.env_id_base, self.env_id_base + self.num_envs, dtype=torch.int64),
                "stats": torch.zeros(8, dtype=torch.int64)}

    def load_state_dict(self, sd: dict):
        """Resume from ``state_dict()`` output of any shard layout: the worlds of this handle's global ids, each exactly once."""
        from .sharding import select_shard_records
        rec = select_shard_records(sd, self.env_id_base, self.num_envs, self.fingerprint, 2 + 9 * self.n_entities).numpy()
        self.import_state(rec[:, 2:].reshape(self.num_envs, self.n_entities, 9), rec[:, 0], rec[:, 1])

    def close(self):
        if getattr(self, "_h", None):
            self.lib.wab2_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
