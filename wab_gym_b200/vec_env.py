"""``VecEnv`` — N lockstep Wolves-and-Bushes environments on one B200, device-resident.

The batched counterpart of the reference's ``WolvesAndBushesEnv`` (``/root/reference/wab_env.py:103-342``):
``reset()`` and ``step(actions)`` keep the reference's meaning (same rules, same observation content,
same reward and done) for every environment of the batch, with the auto-reset convention of vector
environments: an environment that reports ``done`` is reset inside the same ``step`` and the
observation returned for it is the first observation of its next episode.

All state lives in HBM behind the C ABI (``include/wab_b200.h``); this class only owns the output
tensors and forwards raw pointers + the current CUDA stream. There is no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Dict, NamedTuple, Optional

import numpy as np
import torch

from . import _lib
from .config import GameConfig

STAT_NAMES = ("episodes", "steps", "finished", "starved", "killed", "eats", "bad_actions", "overflows")


class ObsBatch(NamedTuple):
    """First six elements of the reference's observation tuple (wab_env.py:374-385), batched.

    ``grids[:, 0]`` wolves, ``grids[:, 1]`` bushes, ``grids[:, 2]`` ostriches — u8 one-hot [N, 3, 11, 11]
    indexed ``[5 - dx, 5 - dy]`` like the reference's float64 grids; ``food`` = turns until starvation."""

    grids: torch.Tensor
    food: torch.Tensor
    role: torch.Tensor
    status: torch.Tensor


class EnvStates(NamedTuple):
    """Saved state of n envs (``VecEnv.save_state``): one opaque record per env (layout: ``WAB_STATE_FORMAT`` in
    ``include/wab_b200.h``), the global id each record was saved from, and the fingerprint of the options, seed and
    kernel family the records belong to."""

    records: torch.Tensor      # u8[n, record_bytes] on the device
    env_ids: torch.Tensor      # i64[n] global env ids (CPU)
    fingerprint: int


#: version of the state record layout (WAB_STATE_FORMAT)
STATE_FORMAT = 1

_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)   # the current stream's handle without a Stream object


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


class VecEnv:
    def __init__(self, num_envs: int, game_options: Optional[dict] = None, device="cuda", seed: int = 0,
                 env_id_base: int = 0, auto_reset: bool = True, wolf_cap: int = 16, log_cap: Optional[int] = None,
                 force_f64_food: bool = False, features: bool = False, ego: bool = False, emit_grids: bool = True,
                 replicas: int = 1, blocks: int = 1, block_stride: int = 0):
        self._h = None
        self._bound = None     # feature buffer currently bound in the handle
        self.lib = _lib.load()  # raises if the CUDA library is unavailable — no fallback
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("VecEnv runs on CUDA devices only (got %r)" % (device,))
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._dev_index = self.device.index
        self.num_envs = int(num_envs)
        self.game = game_options if isinstance(game_options, GameConfig) else GameConfig.from_options(
            game_options, auto_reset=auto_reset, force_f64_food=force_f64_food, wolf_cap=wolf_cap, log_cap=log_cap)
        self.game_options = self.game.options
        self.n_actions = self.game.n_actions
        #: viewport (wab_env.py:25-26): grids are u8[N, 3, width, height]; 11 x 11 with spawn margin 1 runs on the
        #: specialised kernels, every other odd size up to 31 x 31 (margins 1, 2) on the warp-per-env generic ones
        self.view = (int(self.game_options["width"]), int(self.game_options["height"]))
        self.seed, self.env_id_base = int(seed), int(env_id_base)
        #: replicas = R > 1: the N envs are R copies of n = N / R envs. Row r has global env id env_id_base + r % n in every
        #: draw keyed by the global id (world, policy noise and samples), so block k, driven by its own actions, plays what
        #: VecEnv(n, env_id_base=env_id_base) plays: R policies can be scored on the same episodes side by side. The ids are
        #: not unique, so state_dict / load_state_dict and load_state without slots refuse such a handle, as do the trainers.
        self.replicas = int(replicas)
        if self.replicas < 1 or self.num_envs % self.replicas != 0:
            raise ValueError("replicas must divide num_envs (got %d envs, %d replicas)" % (self.num_envs, self.replicas))
        #: blocks = K > 1: the N envs are K blocks of c = N / K envs, and row k c + j has global env id env_id_base +
        #: k block_stride + j in every draw keyed by the global id, so block k, driven by its own actions, plays what
        #: VecEnv(c, env_id_base=env_id_base + k block_stride) plays. With block_stride >= c the ids are unique: one handle
        #: holds a shard of every member of a data-parallel population (ids B + p n + first .. of member p). state_dict,
        #: load_state_dict and load_state without slots work on the blocked ids (``global_ids`` / ``slots_of_ids``).
        self.blocks, self.block_stride = int(blocks), int(block_stride)
        if self.blocks > 1 and self.replicas > 1:
            raise ValueError("a handle has replicas or blocks, not both")
        if self.blocks < 1 or self.num_envs % self.blocks != 0:
            raise ValueError("blocks must divide num_envs (got %d envs, %d blocks)" % (self.num_envs, self.blocks))
        if self.blocks > 1 and self.block_stride < self.num_envs // self.blocks:
            raise ValueError("block_stride must be at least num_envs / blocks = %d, or the blocks' ids overlap (got %d)"
                             % (self.num_envs // self.blocks, self.block_stride))
        cs = self.game.to_struct()
        thr = np.ascontiguousarray(self.game.bush_thr, dtype=np.uint32)
        handle = ctypes.c_void_p()
        _lib.check(self.lib.wab_vec_create(ctypes.byref(cs), thr.ctypes.data, len(thr), self.num_envs,
                                           self.seed & 0xFFFFFFFFFFFFFFFF, self.env_id_base, self.device.index,
                                           ctypes.byref(handle)))
        self._h = handle
        if self.replicas > 1:
            _lib.check(self.lib.wab_vec_set_replicas(self._h, self.replicas))
        if self.blocks > 1:
            _lib.check(self.lib.wab_vec_set_blocks(self._h, self.blocks, self.block_stride))
        self.lanes_per_env = int(self.lib.wab_vec_lanes_per_env(self._h))
        self.generic_kernels = bool(self.lib.wab_vec_kernel_kind(self._h))
        self.with_ego = bool(ego)
        if ego:      # egocentric observation family: the kernels keep every episode's position history
            _lib.check(self.lib.wab_vec_enable_ego(self._h))
        self.with_features = bool(features)
        #: emit_grids=False (needs features=True): FEATURES-ONLY stepping — the kernels write the 28 PragmaticObsWrapper bytes,
        #: scalars, reward, done and info per env and never materialise the 363-byte one-hot grids (ObsBatch.grids is None):
        #: what the reference's actor-critic consumes (actor_critic.py:42, :188) at a thirteenth of the output traffic
        self.emit_grids = bool(emit_grids)
        if not self.emit_grids and (not self.with_features or self.generic_kernels):
            raise ValueError("emit_grids=False needs features=True and the default 11 x 11 viewport")
        self.flat_dim = int(self.lib.wab_vec_flat_dim(self._h))
        #: bytes of one env's state record and the fingerprint records must carry to load here (save_state / load_state)
        self.record_bytes = int(self.lib.wab_vec_state_record_bytes(self._h))
        fp = ctypes.c_uint64()
        _lib.check(self.lib.wab_vec_state_fingerprint(self._h, ctypes.byref(fp)))
        self.fingerprint = int(fp.value)
        self._out = self._alloc(None)
        self._many: Dict[int, dict] = {}

    # ------------------------------------------------------------------ buffers
    def _alloc(self, steps: Optional[int]) -> dict:
        n, dev = self.num_envs, self.device
        lead = (n,) if steps is None else (steps, n)
        u8 = dict(dtype=torch.uint8, device=dev)
        extra = {"features": torch.empty(lead + (28,), **u8)} if self.with_features else {}
        return {
            **extra,
            "grids": torch.empty(lead + (3,) + self.view, **u8) if self.emit_grids else None, "food": torch.empty(lead, **u8),
            "role": torch.empty(lead, **u8), "status": torch.empty(lead, **u8),
            "reward": torch.empty(lead, dtype=torch.float32, device=dev), "done": torch.empty(lead, **u8),
            "info": torch.empty(lead, **u8),
        }

    @staticmethod
    def _obs_struct(buf) -> _lib.WabObs:
        return _lib.WabObs(buf["grids"].data_ptr() if buf.get("grids") is not None else 0, buf["food"].data_ptr(),
                           buf["role"].data_ptr(), buf["status"].data_ptr())

    def _bind(self, buf):
        """Point the fused PragmaticObsWrapper feature output at this call's buffer (or switch it off)."""
        f = buf.get("features")
        self._bound = f
        _lib.check(self.lib.wab_vec_bind_features(self._h, _ptr(f)))

    def _info(self, buf):
        info = {"info": buf["info"]}
        if "features" in buf:
            info["features"] = buf["features"]
        return info

    def _stream(self):
        if _raw_stream is not None:
            return ctypes.c_void_p(_raw_stream(self._dev_index))
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _actions_u8(self, actions: torch.Tensor, shape) -> torch.Tensor:
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(actions)
        if tuple(actions.shape) != tuple(shape):
            raise ValueError("actions must have shape %r, got %r" % (tuple(shape), tuple(actions.shape)))
        if actions.device != self.device:
            actions = actions.to(self.device, non_blocking=True)
        if actions.dtype != torch.uint8:
            # the reference raises IndexError for anything outside 0..n_actions-1 (wab_env.py:253); a batch cannot, so
            # such values become 255 — a bad action: the env does not move and stats()['bad_actions'] counts it —
            # BEFORE the narrowing cast (which would otherwise wrap 256 to 0, -252 to 4, ...)
            if actions.dtype.is_floating_point or actions.dtype == torch.bool:
                raise TypeError("actions must be an integer tensor")
            actions = torch.where((actions < 0) | (actions >= self.n_actions), 255, actions).to(torch.uint8)
        return actions.contiguous()

    # ------------------------------------------------------------------ gym-like surface
    def reset(self, mask: Optional[torch.Tensor] = None) -> ObsBatch:
        """reset() of the reference (wab_env.py:231-248) for every env (or those with ``mask != 0``)."""
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if mask.shape != (self.num_envs,):
                raise ValueError("mask must have shape (num_envs,)")
        b = self._out
        self._bind(b)
        _lib.check(self.lib.wab_vec_reset(self._h, _ptr(mask), self._obs_struct(b), self._stream()))
        return ObsBatch(b["grids"], b["food"], b["role"], b["status"])

    def step(self, actions: torch.Tensor):
        """step(action) of the reference (wab_env.py:250-342) for every env. Returns
        ``(ObsBatch, reward f32[N], done bool[N], info)``; tensors are reused by the next call."""
        a = self._actions_u8(actions, (self.num_envs,))
        b = self._out
        self._bind(b)
        _lib.check(self.lib.wab_vec_step(self._h, _ptr(a), self._obs_struct(b), _ptr(b["reward"]), _ptr(b["done"]),
                                         _ptr(b["info"]), self._stream()))
        return (ObsBatch(b["grids"], b["food"], b["role"], b["status"]), b["reward"], b["done"].view(torch.bool),
                self._info(b))

    def step_kernel_name(self, n_steps=1):
        """The kernel a launch of `n_steps` lockstep steps runs (benchmarks and profiles name it)."""
        if self.generic_kernels:
            return "wab_generic_step_kernel"
        if self.lib.wab_vec_step_many_pipelined(self._h, int(n_steps)):
            return "wab_step_pipe_kernel<false, LPE=%d> (rule warp + publisher warp per env group)" % self.lanes_per_env
        return "wab_step_kernel<false, LPE=%d>" % self.lanes_per_env

    def step_many(self, actions: torch.Tensor, out: Optional[dict] = None):
        """T lockstep steps in one launch; ``actions`` u8[T, N]. Every step's observation, reward and
        done are materialised ([T, N, ...]); state stays in registers between steps."""
        steps = int(actions.shape[0])
        a = self._actions_u8(actions, (steps, self.num_envs))
        b = out if out is not None else self._many.get(steps)
        if b is None:
            b = self._many[steps] = self._alloc(steps)
        self._bind(b)
        _lib.check(self.lib.wab_vec_step_many(self._h, steps, _ptr(a), self._obs_struct(b), _ptr(b["reward"]),
                                              _ptr(b["done"]), _ptr(b["info"]), self._stream()))
        return (ObsBatch(b["grids"], b["food"], b["role"], b["status"]), b["reward"], b["done"].view(torch.bool),
                self._info(b))

    # ------------------------------------------------------------------ PragmaticObsWrapper on the device
    @property
    def last_features(self) -> Optional[torch.Tensor]:
        """u8[N, 28] features of the observation returned by the last reset()/step() (features=True)."""
        return self._out.get("features")

    def pragmatic_features(self, obs: ObsBatch) -> torch.Tensor:
        """PragmaticObsWrapper.observation (wab_env.py:726-761) for any observation batch: u8[..., 28] =
        nearest_wolf[4] second_wolf[4] n_wolves[4] nearest_bush[4] second_bush[4] n_bushes[4] standing food role status."""
        lead = obs.food.shape
        out = torch.empty(lead + (28,), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.wab_pragmatic_features(_ptr(obs.grids.contiguous()), _ptr(obs.food.contiguous()),
                                                   _ptr(obs.role.contiguous()), _ptr(obs.status.contiguous()),
                                                   obs.food.numel(), _ptr(out), self._stream()))
        return out

    def flatten_features(self, features: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """gym.spaces.flatten of the wrapper observation (actor_critic.py:188): f32[..., flat_dim] one-hot
        (449 columns under default options), including the role's view mask."""
        features = features.contiguous()
        lead = features.shape[:-1]
        if out is None:
            out = torch.empty(lead + (self.flat_dim,), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.wab_vec_flatten_features(self._h, _ptr(features), features.numel() // 28, _ptr(out),
                                                     self._stream()))
        return out

    def flatten_features_noisy(self, features: torch.Tensor, out: torch.Tensor, noise_scale: float = 0.01,
                               counter: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The policy input of ``actor_critic.py:188-189`` in one kernel: flatten + ``noise_scale * U[0,1)`` + cast to
        ``out.dtype`` (float32 or bfloat16). ``counter`` is an int64[1] device tensor the caller advances between
        calls (fresh noise per call, also under CUDA-graph replay)."""
        features = features.contiguous()
        rows = features.numel() // 28
        if out.dtype not in (torch.float32, torch.bfloat16) or out.numel() != rows * self.flat_dim or not out.is_contiguous():
            raise ValueError("out must be a contiguous float32 or bfloat16 tensor of rows x flat_dim elements")
        _lib.check(self.lib.wab_vec_flatten_features_noisy(self._h, _ptr(features), rows, _ptr(out),
                                                           int(out.dtype == torch.bfloat16), float(noise_scale),
                                                           _ptr(counter), self._stream()))
        return out

    def sample_actions(self, probs: torch.Tensor, out: torch.Tensor, counter: Optional[torch.Tensor] = None,
                       seed: int = 0) -> torch.Tensor:
        """``Categorical(probs).sample()`` (``actor_critic.py:117-120``) for every row of ``probs`` ([N, A], float32 or
        bfloat16, A <= 8) into the uint8 tensor ``out`` — one small kernel instead of torch.multinomial."""
        probs = probs.contiguous()
        if probs.dtype not in (torch.float32, torch.bfloat16) or out.dtype != torch.uint8 or out.numel() != probs.shape[0]:
            raise ValueError("probs must be float32/bfloat16 [N, A] and out uint8[N]")
        _lib.check(self.lib.wab_sample_categorical(_ptr(probs), int(probs.dtype == torch.bfloat16), probs.shape[0],
                                                   probs.shape[1], int(seed) & (2 ** 64 - 1), _ptr(counter), _ptr(out),
                                                   self._stream()))
        return out

    def ego_proximities(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The reference's egocentric observations (``_get_wolf_proximities`` / ``_get_bush_proximities``,
        wab_env.py:637-667) of the state left by the last reset()/step(): u8[N, 10] = wolves[5], bushes[5] for the
        squares up, right, down, left, stay; ``WolvesAndBushesEnvEgoCentric._get_obs`` (:951-958) is
        ``(out[:, 5:], food, role, status)``. Needs ``VecEnv(ego=True)``."""
        if not self.with_ego:
            raise ValueError("ego_proximities needs VecEnv(ego=True)")
        if out is None:
            out = torch.empty((self.num_envs, 10), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.wab_vec_ego_proximities(self._h, _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ host-buffer entry points
    def alloc_host_buffers(self, pinned: bool = True) -> dict:
        """Host-side buffers for the host entry points: every output is a view into ONE (pinned) block laid out by
        ``wab_vec_host_block_layout`` so a step needs a single device-to-host transfer."""
        n = self.num_envs
        offs = np.zeros(7, dtype=np.int64)
        total = ctypes.c_int64()
        _lib.check(self.lib.wab_vec_host_block_layout(self._h, offs.ctypes.data, ctypes.addressof(total)))
        block = torch.empty(total.value, dtype=torch.uint8, pin_memory=pinned)
        view = lambda k, nbytes: block[int(offs[k]):int(offs[k]) + nbytes]
        hb = {"actions": torch.empty(n, dtype=torch.uint8, pin_memory=pinned), "block": block,
              "grids": view(0, n * 3 * self.view[0] * self.view[1]).view(n, 3, *self.view), "food": view(1, n), "role": view(2, n),
              "status": view(3, n),
              "reward": view(4, 4 * n).view(torch.float32), "done": view(5, n), "info": view(6, n)}
        # numpy views of the same memory (cheap per-step access from Python) and the two pointers a step passes
        hb["np"] = {k: v.numpy() for k, v in hb.items() if k != "block"}
        hb["_c"] = (_ptr(hb["actions"]), _ptr(block))
        return hb

    def step_host(self, hb: dict):
        """One step with HOST buffers (``hb`` from ``alloc_host_buffers``; ``hb['actions']`` filled by the
        caller): H2D actions, kernel, D2H of every output, stream sync — the whole C-ABI host path."""
        if self._bound is not None:
            self._bind({})
        if "_c" in hb:
            rc = self.lib.wab_vec_step_host_packed(self._h, hb["_c"][0], hb["_c"][1], self._stream())
            if rc:
                _lib.check(rc)
        elif "block" in hb:
            _lib.check(self.lib.wab_vec_step_host_packed(self._h, _ptr(hb["actions"]), _ptr(hb["block"]), self._stream()))
        else:
            _lib.check(self.lib.wab_vec_step_host(self._h, _ptr(hb["actions"]), _ptr(hb["grids"]), _ptr(hb["food"]),
                                                  _ptr(hb["role"]), _ptr(hb["status"]), _ptr(hb["reward"]),
                                                  _ptr(hb["done"]), _ptr(hb["info"]), self._stream()))
        return hb

    def free_host_buffers(self, hb: dict):
        """Drop host buffers from ``alloc_host_buffers``: the library forgets what it cached for their addresses (device
        aliases of the pinned block, the captured host-step graph) before the memory goes back to the allocator."""
        _lib.check(self.lib.wab_vec_forget_host_buffers(self._h))
        hb.clear()

    def reset_host(self, hb: dict):
        self._bind({})
        _lib.check(self.lib.wab_vec_reset_host(self._h, _ptr(hb["grids"]), _ptr(hb["food"]), _ptr(hb["role"]),
                                               _ptr(hb["status"]), self._stream()))
        return hb

    # ------------------------------------------------------------------ statistics / introspection
    def stats(self, clear: bool = False) -> Dict[str, int]:
        out = np.zeros(8, dtype=np.int64)
        _lib.check(self.lib.wab_vec_stats(self._h, out.ctypes.data, int(clear), self._stream()))
        return dict(zip(STAT_NAMES, (int(v) for v in out)))

    def stats_tensor(self) -> torch.Tensor:
        """int64[8] on the device, enqueued on the current stream (feed to an NCCL all_reduce)."""
        t = torch.empty(8, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.wab_vec_stats_device(self._h, _ptr(t), self._stream()))
        return t

    def export_state(self) -> Dict[str, np.ndarray]:
        n, wc, lc = self.num_envs, self.game.wolf_cap, self.game.log_cap
        i32 = lambda *s: np.zeros(s, dtype=np.int32)
        st = {"x": i32(n), "y": i32(n), "food": np.zeros(n, dtype=np.float64), "role": i32(n), "status": i32(n),
              "turn": i32(n), "episode": np.zeros(n, dtype=np.int64), "n_wolves": i32(n), "wolves": i32(n, wc, 2),
              "bush_mask": np.zeros((n, 4), dtype=np.uint32), "n_log": i32(n), "log": i32(n, lc, 3)}
        order = ("x", "y", "food", "role", "status", "turn", "episode", "n_wolves", "wolves", "bush_mask", "n_log", "log")
        _lib.check(self.lib.wab_vec_export_state(self._h, *(ctypes.c_void_p(st[k].ctypes.data) for k in order),
                                                 self._stream()))
        return st

    # ------------------------------------------------------------------ checkpoint / resume / clone
    def _local_slots(self, slots) -> torch.Tensor:
        s = torch.as_tensor(slots, dtype=torch.int64).reshape(-1).cpu()
        if s.numel() and (int(s.min()) < 0 or int(s.max()) >= self.num_envs):
            raise ValueError("slots must lie in [0, %d)" % self.num_envs)
        return s

    def _layout(self):
        """(blocks, envs per block, block_stride) of this handle's id map: (1, N, 0) for a plain handle, (R, N / R, 0) with
        replicas."""
        if self.replicas > 1:
            return self.replicas, self.num_envs // self.replicas, 0
        if self.blocks > 1:
            return self.blocks, self.num_envs // self.blocks, self.block_stride
        return 1, self.num_envs, 0

    def global_ids(self, slots=None) -> torch.Tensor:
        """The global env id of every slot (or of ``slots``), int64 on the CPU: the key of every draw made for it."""
        local = torch.arange(self.num_envs, dtype=torch.int64) if slots is None else self._local_slots(slots)
        from .sharding import blocked_env_ids
        return blocked_env_ids(local, *self._layout(), self.env_id_base)

    def slots_of_ids(self, env_ids) -> torch.Tensor:
        """The slot of every global id of ``env_ids`` (int64, CPU). Raises ``ValueError`` for an id this handle does not
        hold, or on a handle with replicas, whose ids repeat."""
        self._refuse_replicas("slots_of_ids")
        from .sharding import blocked_env_slots
        return blocked_env_slots(torch.as_tensor(env_ids, dtype=torch.int64).reshape(-1).cpu(), *self._layout(),
                                 self.env_id_base)

    def save_state(self, slots=None) -> EnvStates:
        """The state of every env (or of ``slots``, in that order) as records on the device. Enqueued on the current
        stream; nothing synchronises. On a handle with replicas the ids repeat: block k's records carry block 0's ids. On a
        blocked handle they are the blocked ids."""
        if slots is None:
            local, d_slots = torch.arange(self.num_envs, dtype=torch.int64), None
        else:
            local = self._local_slots(slots)
            d_slots = local.to(device=self.device, dtype=torch.int32)
        records = torch.empty((local.numel(), self.record_bytes), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.wab_vec_save_state(self._h, _ptr(d_slots), local.numel(), _ptr(records), self._stream()))
        from .sharding import blocked_env_ids
        return EnvStates(records, blocked_env_ids(local, *self._layout(), self.env_id_base), self.fingerprint)

    def load_state(self, states: EnvStates, slots=None) -> ObsBatch:
        """Write each record of ``states`` into a slot: the slot of its own global id (which must belong to this handle),
        or ``slots[r]`` — a clone of the saved env whose future draws are keyed by the destination's global id. Every
        check passes before anything is written; a refused load raises ``ValueError`` and changes nothing. Returns the
        observation of every env, as ``reset`` with an empty mask would (``last_features`` is updated too). Synchronises
        once, to read the device-side verdict."""
        if slots is None and self.replicas > 1:
            raise ValueError("a handle with replicas repeats its env ids: load_state needs slots")
        records = states.records
        if records.dtype != torch.uint8 or records.dim() != 2 or records.shape[1] != self.record_bytes:
            raise ValueError("records must be uint8 [n, %d] for this handle" % self.record_bytes)
        if int(states.fingerprint) != self.fingerprint:
            raise ValueError("state fingerprint %#x does not match this handle (%#x): different options, seed, wolf/log caps, "
                             "kernel family or ego setting" % (int(states.fingerprint), self.fingerprint))
        n = records.shape[0]
        if slots is None:
            ids = torch.as_tensor(states.env_ids, dtype=torch.int64).reshape(-1).cpu()
            if ids.numel() != n:
                raise ValueError("env_ids and records disagree in length")
            local = self.slots_of_ids(ids)
        else:
            local = self._local_slots(slots)
            if local.numel() != n:
                raise ValueError("slots and records disagree in length")
        if torch.unique(local).numel() != n:
            raise ValueError("duplicate destination slots")
        identity = n == self.num_envs and torch.equal(local, torch.arange(n, dtype=torch.int64))
        d_slots = None if identity else local.to(device=self.device, dtype=torch.int32)
        records = records.to(self.device).contiguous()
        rejected = torch.zeros(1, dtype=torch.int32, device=self.device)
        b = self._out
        self._bind(b)
        _lib.check(self.lib.wab_vec_load_state(self._h, _ptr(records), _ptr(d_slots), n, self._obs_struct(b), _ptr(rejected),
                                               self._stream()))
        bad = int(rejected.item())
        if bad:
            raise ValueError("%d of %d state records refused (format word, fingerprint, or a wolf count, log length, role, "
                             "status, food or turn outside what the kernels maintain); nothing was loaded" % (bad, n))
        return ObsBatch(b["grids"], b["food"], b["role"], b["status"])

    def state_dict(self) -> dict:
        """Everything a resume needs, on the host (``torch.save`` works): format, fingerprint, global env ids, the records
        and the 8 statistics totals. ``sharding.merge_state_dicts`` joins the dicts of several shards."""
        self._refuse_replicas("state_dict")
        st = self.save_state()
        stats = self.stats()
        return {"format": STATE_FORMAT, "fingerprint": st.fingerprint, "env_ids": st.env_ids.clone(),
                "records": st.records.cpu(), "stats": torch.tensor([stats[k] for k in STAT_NAMES], dtype=torch.int64)}

    def load_state_dict(self, sd: dict) -> ObsBatch:
        """Resume from ``state_dict()`` output (of this or any other shard layout: the records of this handle's global ids
        are picked, each exactly once; on a blocked handle each block's range). The statistics totals go to the shard
        holding env 0 and every other shard starts from zero, so their sum is preserved."""
        self._refuse_replicas("load_state_dict")
        from .sharding import select_shard_records
        K, c, stride = self._layout()
        records = torch.cat([select_shard_records(sd, self.env_id_base + k * stride, c, self.fingerprint, self.record_bytes)
                             for k in range(K)])            # block k: its contiguous id range, in slot order
        obs = self.load_state(EnvStates(records, self.global_ids(), self.fingerprint))
        stats = np.zeros(8, dtype=np.int64)
        if self.env_id_base == 0:
            stats[:] = torch.as_tensor(sd["stats"], dtype=torch.int64).numpy()
        _lib.check(self.lib.wab_vec_set_stats(self._h, stats.ctypes.data, self._stream()))
        return obs

    def _refuse_replicas(self, what: str):
        if self.replicas > 1:
            raise ValueError("%s needs unique env ids; this handle has %d replicas (use save_state / load_state with slots)"
                             % (what, self.replicas))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.wab_vec_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
