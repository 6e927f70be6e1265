"""Actor-critic policy and device-resident rollout (BASELINE config 5).

The reference's consumer of the environment is ``actor_critic.py``: a 4-layer MLP
(``Policy``, ``actor_critic.py:54-97``) fed with ``gym.spaces.flatten`` of the ``PragmaticObsWrapper``
observation plus ``U[0,1)/100`` input noise (``:188-189``), a ``Categorical`` sample per step (``:108-125``,
with a host sync per step through ``.item()``), stepping ONE environment. Here the same network
consumes the flattened features of N environments straight from HBM: features and the 449-column
one-hot come from the CUDA kernels (``wab_features.cuh``), the MLP is plain torch (cuBLAS GEMMs — a
library GEMM, not a hot op of this path), sampling stays on the device and nothing synchronises with
the host inside the loop.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd.function import once_differentiable

from . import _lib
from .vec_env import VecEnv, _ptr, _raw_stream


class Policy(nn.Module):
    """Same architecture as the reference's ``Policy`` (``actor_critic.py:54-97``)."""

    def __init__(self, obs_dim: int, n_actions: int):
        super().__init__()
        self.affine1 = nn.Linear(obs_dim, 128)
        self.affine2 = nn.Linear(128, 150)
        self.affine3 = nn.Linear(150, 128)
        self.action_head = nn.Linear(128, n_actions)
        self.value_head = nn.Linear(128, 1)

    def forward(self, x):
        x = F.leaky_relu(self.affine1(x))
        x = F.leaky_relu(self.affine2(x))
        x = F.leaky_relu(self.affine3(x))
        x = torch.clamp(x, -4, 4)
        return F.softmax(self.action_head(x), dim=-1), self.value_head(x)


def policy_tail(policy: "Policy", z3: torch.Tensor, heads: tuple, actions: torch.Tensor, value: Optional[torch.Tensor] = None,
                probs: Optional[torch.Tensor] = None, logp: Optional[torch.Tensor] = None,
                counter: Optional[torch.Tensor] = None, seed: int = 0) -> torch.Tensor:
    """``clamp(leaky_relu(z3)) -> action_head / value_head -> softmax -> Categorical.sample()`` (``actor_critic.py:92-97``,
    ``:114-120``) as ONE kernel of the library (``wab_policy_tail``): ``z3`` f32[N, 128] is ``policy.affine3``'s output
    before its activation, ``heads`` = ``stacked_heads(policy)``. Fills ``actions`` u8[N] (and ``value``, ``probs``,
    ``logp`` when given)."""
    w, b = heads
    if z3.dtype != torch.float32 or not z3.is_contiguous() or z3.shape[1] != 128:
        raise ValueError("z3 must be a contiguous float32 [N, 128] tensor")
    dev = z3.device.index if z3.device.index is not None else torch.cuda.current_device()
    stream = ctypes.c_void_p(_raw_stream(dev)) if _raw_stream is not None else ctypes.c_void_p(torch.cuda.current_stream(z3.device).cuda_stream)
    _lib.check(_lib.load().wab_policy_tail(_ptr(z3), 128, _ptr(w), _ptr(b), z3.shape[0], w.shape[0] - 1, 0.01, -4.0, 4.0,
                                           int(seed) & (2 ** 64 - 1), _ptr(counter), _ptr(actions), _ptr(value), _ptr(probs),
                                           _ptr(logp), stream))
    return actions


def check_reference_network(policy: "Policy", flat_dim: int, who: str) -> None:
    """What the tensor-core policy kernels serve: the reference's network (``flat_dim -> 128 -> 150 -> 128 -> {A <= 8, 1}``)
    in fp32. Raises ``ValueError`` naming ``who`` otherwise; reads shapes and dtypes only."""
    p = policy
    if any(prm.dtype != torch.float32 for prm in p.parameters()):
        raise ValueError("%s needs an fp32 policy" % who)
    shapes = [(m.in_features, m.out_features) for m in (p.affine1, p.affine2, p.affine3, p.value_head)]
    if shapes != [(flat_dim, 128), (128, 150), (150, 128), (128, 1)] or p.action_head.in_features != 128 or \
            not 1 <= p.action_head.out_features <= 8:
        raise ValueError("%s is built for the reference's network: flat_dim -> 128 -> 150 -> 128 -> {A <= 8, 1}" % who)


def stacked_heads(policy: "Policy") -> tuple:
    """(action_head.weight stacked on value_head.weight f32[A + 1, 128], the two biases f32[A + 1]) — refresh after an
    optimiser step."""
    with torch.no_grad():
        w = torch.cat([policy.action_head.weight, policy.value_head.weight], 0).float().contiguous()
        b = torch.cat([policy.action_head.bias, policy.value_head.bias], 0).float().contiguous()
    return w, b


class Affine1TC:
    """``leaky_relu(policy.affine1(flatten(obs) + noise))`` (``actor_critic.py:59``, ``:88-90``, ``:188-189``) as ONE tcgen05
    kernel of the library (``wab_policy_affine1``): the 449-wide input is generated inside the kernel from the 28 feature
    bytes per environment — same keyed noise as ``VecEnv.flatten_features_noisy`` — and the product runs on the tensor
    cores with bf16 x 3 operand splits and fp32 accumulation, i.e. to fp32 accuracy. ``refresh()`` re-packs the weights
    after an optimiser step."""

    def __init__(self, env: VecEnv, policy: "Policy"):
        if policy.affine1.out_features != 128 or policy.affine1.in_features != env.flat_dim:
            raise ValueError("Affine1TC is built for the reference's affine1: flat_dim -> 128")
        self.env, self.policy, self.lib = env, policy, _lib.load()
        self.packed = torch.empty(int(self.lib.wab_policy_affine1_packed_bytes()), dtype=torch.uint8, device=env.device)
        self.bias = None
        self.refresh()

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream)

    @torch.no_grad()
    def refresh(self):
        w = self.policy.affine1.weight.detach().float().contiguous()
        b = self.policy.affine1.bias.detach().float().contiguous()
        self.bias = b.clone() if self.bias is None else self.bias.copy_(b)           # in place: captured graphs hold the pointer
        _lib.check(self.lib.wab_policy_affine1_prepare(_ptr(w), w.shape[1], _ptr(self.packed), self._stream()))

    def __call__(self, features: torch.Tensor, out: torch.Tensor, noise_scale: float = 0.01,
                 counter: Optional[torch.Tensor] = None, slope: float = 0.01) -> torch.Tensor:
        if out.dtype != torch.float32 or not out.is_contiguous() or tuple(out.shape) != (features.shape[0], 128):
            raise ValueError("out must be a contiguous float32 [N, 128] tensor")
        _lib.check(self.lib.wab_policy_affine1(self.env._h, _ptr(features), features.shape[0], _ptr(self.packed), _ptr(self.bias),
                                               float(noise_scale), float(slope), _ptr(counter), _ptr(out), self._stream()))
        return out


class PolicyTrunkTC(Affine1TC):
    """The whole trunk ``affine3(leaky_relu(affine2(leaky_relu(affine1(flatten(obs) + noise)))))`` (``actor_critic.py:88-92``)
    as ONE tcgen05 kernel (``wab_policy_trunk``): returns ``z3`` f32[N, 128], the pre-activation output of ``affine3`` that
    ``policy_tail`` takes. The hidden activations never leave the SM."""

    def __init__(self, env: VecEnv, policy: "Policy"):
        if (policy.affine2.in_features, policy.affine2.out_features, policy.affine3.in_features, policy.affine3.out_features) != (128, 150, 150, 128):
            raise ValueError("PolicyTrunkTC is built for the reference's trunk: 128 -> 150 -> 128")
        lib = _lib.load()
        self.packed2 = torch.empty(int(lib.wab_policy_linear_packed_bytes(150, 128)), dtype=torch.uint8, device=env.device)
        self.packed3 = torch.empty(int(lib.wab_policy_linear_packed_bytes(128, 150)), dtype=torch.uint8, device=env.device)
        self.bias2 = self.bias3 = None
        super().__init__(env, policy)

    @torch.no_grad()
    def refresh(self):
        super().refresh()
        p = self.policy
        w2, w3 = p.affine2.weight.detach().float().contiguous(), p.affine3.weight.detach().float().contiguous()
        b2, b3 = p.affine2.bias.detach().float().contiguous(), p.affine3.bias.detach().float().contiguous()
        self.bias2 = b2.clone() if self.bias2 is None else self.bias2.copy_(b2)
        self.bias3 = b3.clone() if self.bias3 is None else self.bias3.copy_(b3)
        _lib.check(self.lib.wab_policy_linear_prepare(_ptr(w2), 150, 128, _ptr(self.packed2), self._stream()))
        _lib.check(self.lib.wab_policy_linear_prepare(_ptr(w3), 128, 150, _ptr(self.packed3), self._stream()))

    def __call__(self, features: torch.Tensor, out: torch.Tensor, noise_scale: float = 0.01,
                 counter: Optional[torch.Tensor] = None, slope: float = 0.01) -> torch.Tensor:
        if out.dtype != torch.float32 or not out.is_contiguous() or tuple(out.shape) != (features.shape[0], 128):
            raise ValueError("out must be a contiguous float32 [N, 128] tensor")
        _lib.check(self.lib.wab_policy_trunk(self.env._h, _ptr(features), features.shape[0], _ptr(self.packed), _ptr(self.bias),
                                             _ptr(self.packed2), _ptr(self.bias2), 150, _ptr(self.packed3), _ptr(self.bias3),
                                             float(noise_scale), float(slope), _ptr(counter), _ptr(out), self._stream()))
        return out


    def forward_sample(self, features: torch.Tensor, heads: tuple, actions: torch.Tensor, value: Optional[torch.Tensor] = None,
                       probs: Optional[torch.Tensor] = None, logp: Optional[torch.Tensor] = None, noise_scale: float = 0.01,
                       counter: Optional[torch.Tensor] = None, seed: int = 0, z3: Optional[torch.Tensor] = None,
                       slope: float = 0.01) -> torch.Tensor:
        """``Policy.forward`` + ``select_action`` (``actor_critic.py:84-97``, ``:108-125``) in ONE launch (``wab_policy_forward``):
        the trunk above, then clamp, both heads, softmax and the Categorical sample of ``policy_tail`` on the accumulators'
        registers. ``heads`` = ``stacked_heads(policy)``; fills ``actions`` u8[N] (and ``value``, ``probs``, ``logp``, ``z3`` when given)."""
        w, b = heads
        _lib.check(self.lib.wab_policy_forward(self.env._h, _ptr(features), features.shape[0], _ptr(self.packed), _ptr(self.bias),
                                               _ptr(self.packed2), _ptr(self.bias2), 150, _ptr(self.packed3), _ptr(self.bias3),
                                               _ptr(w), _ptr(b), w.shape[0] - 1, float(noise_scale), float(slope), -4.0, 4.0,
                                               int(seed) & (2 ** 64 - 1), _ptr(counter), _ptr(actions), _ptr(value), _ptr(probs),
                                               _ptr(logp), _ptr(z3), self._stream()))
        return actions

    def forward_greedy(self, features: torch.Tensor, heads: tuple, actions: torch.Tensor, value: Optional[torch.Tensor] = None,
                       probs: Optional[torch.Tensor] = None, logp: Optional[torch.Tensor] = None, noise_scale: float = 0.01,
                       counter: Optional[torch.Tensor] = None, z3: Optional[torch.Tensor] = None,
                       slope: float = 0.01) -> torch.Tensor:
        """``forward_sample`` with the deterministic action in place of the sample, in ONE launch (``wab_policy_act``):
        ``actions`` u8[N] = the first index of the largest logit, ``torch.argmax`` of the action head's output. ``value``
        and ``probs`` are ``forward_sample``'s bit for bit, ``logp`` is the log-probability of the greedy action. The input
        noise is unchanged (``noise_scale=0``: the argmax of the bare network)."""
        w, b = heads
        _lib.check(self.lib.wab_policy_act(self.env._h, _ptr(features), features.shape[0], _ptr(self.packed), _ptr(self.bias),
                                           _ptr(self.packed2), _ptr(self.bias2), 150, _ptr(self.packed3), _ptr(self.bias3),
                                           _ptr(w), _ptr(b), w.shape[0] - 1, float(noise_scale), float(slope), -4.0, 4.0,
                                           _ptr(counter), _ptr(actions), _ptr(value), _ptr(probs), _ptr(logp), _ptr(z3),
                                           self._stream()))
        return actions


class PolicyTrainTC(PolicyTrunkTC):
    """The backward pass of ``Policy.forward`` on the tensor cores (``wab_policy_backward``): from what a rollout with
    ``forward_sample`` recorded — features u8[T, N, 28], the noise counter of each step int64[T], actions u8[T, N] — and
    upstream gradients ``g_logp``, ``g_value`` f32[T, N] of the sampled actions' log-probabilities and of the values, the
    gradient of ``sum g_logp * log pi(a | x) + g_value * V(x)`` with respect to every parameter of the policy, as one flat
    f32 buffer in ``parameters_to_vector(policy.parameters())`` order. The forward is recomputed from the feature bytes
    (the policy input is regenerated, never stored), so training keeps 62 bytes per env-step instead of autograd's
    activations. ``refresh()`` after an optimiser step re-packs the weights, the transposed ones included.

    ``logits_and_value`` is the same pass behind autograd, for any loss written in torch: it refreshes by itself."""

    def __init__(self, env: VecEnv, policy: "Policy"):
        lib = _lib.load()
        self.packed2t = torch.empty(int(lib.wab_policy_linear_packed_bytes(128, 150)), dtype=torch.uint8, device=env.device)
        self.packed3t = torch.empty(int(lib.wab_policy_linear_packed_bytes(150, 128)), dtype=torch.uint8, device=env.device)
        self.scratch = torch.empty(int(lib.wab_policy_backward_scratch_bytes(env._h)), dtype=torch.uint8, device=env.device)
        self.heads = None
        super().__init__(env, policy)
        if policy.action_head.weight.shape[0] > 8 or policy.action_head.in_features != 128 or policy.value_head.in_features != 128:
            raise ValueError("PolicyTrainTC is built for the reference's heads: 128 -> {A <= 8, 1}")
        self.n_params = sum(p.numel() for p in policy.parameters())

    @torch.no_grad()
    def refresh(self):
        super().refresh()
        p = self.policy
        w2t, w3t = p.affine2.weight.detach().float().t().contiguous(), p.affine3.weight.detach().float().t().contiguous()
        _lib.check(self.lib.wab_policy_linear_prepare(_ptr(w2t), 128, 150, _ptr(self.packed2t), self._stream()))
        _lib.check(self.lib.wab_policy_linear_prepare(_ptr(w3t), 150, 128, _ptr(self.packed3t), self._stream()))
        w, b = stacked_heads(p)
        if self.heads is None:
            self.heads = (w, b)
        else:
            self.heads[0].copy_(w); self.heads[1].copy_(b)
        self._packed_versions = self._versions()

    def _versions(self) -> tuple:
        """The identity and version counter of every parameter: any in-place change (an optimiser step, a load) moves one."""
        return tuple((id(p), p._version) for p in self.policy.parameters())

    def logits_and_value(self, features: torch.Tensor, counters: torch.Tensor, rows: Optional[torch.Tensor] = None,
                         noise_scale: float = 0.01, slope: float = 0.01):
        """The policy's outputs for a list of recorded rows, differentiable with respect to ``policy.parameters()``:
        ``(logits f32[M, A], value f32[M])``, the action head's output before the softmax and the value head's, for the
        rows ``rows`` int32[M] (indices t * N + n into the T * N rows of ``features`` u8[T, N, 28], each under its step's
        counter ``counters`` int64[T]; ``None``: all T * N rows in order). Write any loss of them in torch and call
        ``.backward()``: the gradient comes from one tcgen05 pass that recomputes the forward from the feature bytes
        (``wab_policy_backward_logits``), so only the outputs are kept per row, never the activations.

        The forward is ``wab_policy_evaluate``: under the weights a rollout used, ``value`` equals what ``forward_sample``
        returned bit for bit. A listed entry outside [0, T * N) gives NaN and no gradient; a repeated one counts once per
        occurrence. The packed weights are refreshed when a parameter changed since the last pack (no ``refresh()`` after
        ``optimizer.step()``), and an in-place change between the forward and the backward raises autograd's version
        error. Nothing synchronises with the host. Double backward is not supported."""
        if features.dim() != 3 or features.shape[2] != 28 or features.dtype != torch.uint8 or not features.is_contiguous():
            raise ValueError("features must be a contiguous uint8 [T, N, 28] tensor")
        T, N = features.shape[:2]
        if counters.dtype != torch.int64 or counters.numel() != T or not counters.is_contiguous():
            raise ValueError("counters must be a contiguous int64 tensor of T elements")
        if rows is not None and (rows.dtype != torch.int32 or rows.dim() != 1 or not rows.is_contiguous()):
            raise ValueError("rows must be a contiguous int32 [M] tensor")
        for name, t in (("features", features), ("counters", counters), ("rows", rows)):
            if t is not None and t.device != self.env.device:
                raise ValueError("%s must be on the environment's device" % name)
        params = list(self.policy.parameters())
        if any(p.dtype != torch.float32 or p.device != self.env.device for p in params):
            raise ValueError("the policy's parameters must be float32 on the environment's device")
        if self._packed_versions != self._versions():
            self.refresh()
        return _LogitsAndValue.apply(self, features, counters, rows, float(noise_scale), float(slope), *params)

    def backward(self, features: torch.Tensor, counters: torch.Tensor, actions: torch.Tensor, g_logp: torch.Tensor,
                 g_value: torch.Tensor, out: Optional[torch.Tensor] = None, rows: Optional[torch.Tensor] = None,
                 n_rows: Optional[torch.Tensor] = None, noise_scale: float = 0.01, slope: float = 0.01,
                 logp: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Returns the flat gradient (``out`` f32[n_params] if given). ``rows`` int32 / ``n_rows`` int64[1] on the device:
        only the first ``n_rows`` listed rows (indices into the T * N rows) are computed; ``logp`` / ``value`` f32[T, N]
        receive the recomputed log-probabilities and values of those rows."""
        T, N = actions.shape
        if tuple(features.shape) != (T, N, 28) or features.dtype != torch.uint8 or not features.is_contiguous():
            raise ValueError("features must be a contiguous uint8 [T, N, 28] tensor")
        for name, t in (("g_logp", g_logp), ("g_value", g_value)):
            if t.dtype != torch.float32 or tuple(t.shape) != (T, N) or not t.is_contiguous():
                raise ValueError("%s must be a contiguous float32 [T, N] tensor" % name)
        if counters.dtype != torch.int64 or counters.numel() != T or actions.dtype != torch.uint8 or not actions.is_contiguous():
            raise ValueError("counters must be int64[T], actions a contiguous uint8 [T, N] tensor")
        if (rows is None) != (n_rows is None) or (rows is not None and (rows.dtype != torch.int32 or n_rows.dtype != torch.int64)):
            raise ValueError("rows (int32) and n_rows (int64[1]) go together")
        if out is None:
            out = torch.empty(self.n_params, dtype=torch.float32, device=self.env.device)
        if out.dtype != torch.float32 or out.numel() != self.n_params or not out.is_contiguous():
            raise ValueError("out must be a contiguous float32 tensor of n_params elements")
        w, b = self.heads
        _lib.check(self.lib.wab_policy_backward(
            self.env._h, _ptr(features), T, N, _ptr(counters), _ptr(actions), _ptr(g_logp), _ptr(g_value), _ptr(rows), _ptr(n_rows),
            _ptr(self.packed), _ptr(self.bias), _ptr(self.packed2), _ptr(self.bias2), 150, _ptr(self.packed3), _ptr(self.bias3),
            _ptr(self.packed2t), _ptr(self.packed3t), _ptr(w), _ptr(b), w.shape[0] - 1, float(noise_scale), float(slope), -4.0, 4.0,
            _ptr(self.scratch), self.scratch.numel(), _ptr(out), _ptr(logp), _ptr(value), self._stream()))
        return out

    def ppo_backward(self, features: torch.Tensor, counters: torch.Tensor, actions: torch.Tensor, logp_old: torch.Tensor,
                     advantage: torch.Tensor, target: torch.Tensor, rows: Optional[torch.Tensor], n_rows: Optional[torch.Tensor],
                     clip_eps: float, policy_weight: float, value_weight: float, entropy_weight: float,
                     out: Optional[torch.Tensor] = None, logp: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None,
                     entropy: Optional[torch.Tensor] = None, noise_scale: float = 0.01, slope: float = 0.01) -> torch.Tensor:
        """PPO's clipped objective in the same pass (``wab_policy_ppo_backward``): the gradient of the sum over the listed rows
        of ``-policy_weight * min(r A, clip(r, 1 - clip_eps, 1 + clip_eps) A) + value_weight * (V - R)^2 / 2
        - entropy_weight * H`` with ``r = exp(log pi(a | x) - logp_old)``, ``A = advantage``, ``R = target`` (f32[T, N]) and
        log pi, V, H under the current weights. ``rows`` / ``n_rows`` as for ``backward`` (a minibatch); ``logp``, ``value``,
        ``entropy`` f32[T, N] receive the new log-probabilities, values and entropies of the listed rows."""
        T, N = actions.shape
        if tuple(features.shape) != (T, N, 28) or features.dtype != torch.uint8 or not features.is_contiguous():
            raise ValueError("features must be a contiguous uint8 [T, N, 28] tensor")
        for name, t in (("logp_old", logp_old), ("advantage", advantage), ("target", target)):
            if t.dtype != torch.float32 or tuple(t.shape) != (T, N) or not t.is_contiguous():
                raise ValueError("%s must be a contiguous float32 [T, N] tensor" % name)
        for name, t in (("logp", logp), ("value", value), ("entropy", entropy)):
            if t is not None and (t.dtype != torch.float32 or tuple(t.shape) != (T, N) or not t.is_contiguous()):
                raise ValueError("%s must be a contiguous float32 [T, N] tensor" % name)
        if counters.dtype != torch.int64 or counters.numel() != T or actions.dtype != torch.uint8 or not actions.is_contiguous():
            raise ValueError("counters must be int64[T], actions a contiguous uint8 [T, N] tensor")
        if (rows is None) != (n_rows is None) or (rows is not None and (rows.dtype != torch.int32 or n_rows.dtype != torch.int64)):
            raise ValueError("rows (int32) and n_rows (int64[1]) go together")
        if out is None:
            out = torch.empty(self.n_params, dtype=torch.float32, device=self.env.device)
        if out.dtype != torch.float32 or out.numel() != self.n_params or not out.is_contiguous():
            raise ValueError("out must be a contiguous float32 tensor of n_params elements")
        w, b = self.heads
        _lib.check(self.lib.wab_policy_ppo_backward(
            self.env._h, _ptr(features), T, N, _ptr(counters), _ptr(actions), _ptr(logp_old), _ptr(advantage), _ptr(target),
            _ptr(rows), _ptr(n_rows), _ptr(self.packed), _ptr(self.bias), _ptr(self.packed2), _ptr(self.bias2), 150,
            _ptr(self.packed3), _ptr(self.bias3), _ptr(self.packed2t), _ptr(self.packed3t), _ptr(w), _ptr(b), w.shape[0] - 1,
            float(noise_scale), float(slope), -4.0, 4.0, float(clip_eps), float(policy_weight), float(value_weight),
            float(entropy_weight), _ptr(self.scratch), self.scratch.numel(), _ptr(out), _ptr(logp), _ptr(value), _ptr(entropy),
            self._stream()))
        return out

    def grad_f64(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The gradient of the last ``backward`` / ``ppo_backward`` on this stream as f64[n_params]: the same fixed-order
        fp64 sum over the CTAs, not rounded (``wab_policy_backward_grad_f64``). For a cross-rank sum that rounds once."""
        if out is None:
            out = torch.empty(self.n_params, dtype=torch.float64, device=self.env.device)
        if out.dtype != torch.float64 or out.numel() != self.n_params or not out.is_contiguous():
            raise ValueError("out must be a contiguous float64 tensor of n_params elements")
        _lib.check(self.lib.wab_policy_backward_grad_f64(self.env._h, _ptr(self.scratch), self.scratch.numel(),
                                                         self.heads[0].shape[0] - 1, _ptr(out), self._stream()))
        return out

    def grad_sum_ranks(self, rank_grads: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """fp32 of the fp64 sum over ranks, in rank order, of ``rank_grads`` f64[W, n_params] (``wab_policy_grad_sum_ranks``)."""
        if rank_grads.dtype != torch.float64 or rank_grads.dim() != 2 or rank_grads.shape[1] != self.n_params or \
                not rank_grads.is_contiguous():
            raise ValueError("rank_grads must be a contiguous float64 [W, n_params] tensor")
        if out is None:
            out = torch.empty(self.n_params, dtype=torch.float32, device=self.env.device)
        if out.dtype != torch.float32 or out.numel() != self.n_params or not out.is_contiguous():
            raise ValueError("out must be a contiguous float32 tensor of n_params elements")
        _lib.check(self.lib.wab_policy_grad_sum_ranks(_ptr(rank_grads), rank_grads.shape[0], self.n_params, _ptr(out),
                                                      self._stream()))
        return out


class PolicyPopulationTC:
    """P policies of the reference's network on ONE features-enabled ``VecEnv`` of N = P n envs (1 <= P <= 64, n a
    multiple of 128): member p owns env rows [p n, (p + 1) n), and its weights are packed into row p of stacked buffers
    (``wab_policy_forward_population``, ``wab_policy_ppo_backward_population``). Each call does for every member what
    ``PolicyTrainTC`` does for one policy, in one launch, and member p's outputs equal, bit for bit, those of
    ``PolicyTrainTC`` on ``VecEnv(n, env_id_base=p n)`` (with the same env_id_base shift on this handle; on a blocked
    handle, ``VecEnv(n, env_id_base=`` the block's first id ``)``). A member is
    re-packed when one of its parameters changed since its last pack (an optimiser step, a load), as
    ``PolicyTrainTC.logits_and_value`` does."""

    def __init__(self, env: VecEnv, policies):
        policies = list(policies)
        P, N = len(policies), env.num_envs
        if not 1 <= P <= 64:
            raise ValueError("a population has 1 to 64 members")
        if N % P != 0 or (N // P) % 128 != 0:
            raise ValueError("PolicyPopulationTC needs num_envs = P * n with n a multiple of 128")
        for p in policies:
            check_reference_network(p, env.flat_dim, "PolicyPopulationTC")
        A = policies[0].action_head.out_features
        if any(p.action_head.out_features != A for p in policies):
            raise ValueError("every member of a population has the same action count")
        self.env, self.policies, self.lib = env, policies, _lib.load()
        self.n_members, self.member_envs, self.n_actions = P, N // P, A
        self.n_params = sum(prm.numel() for prm in policies[0].parameters())
        self.grad_stride = int(self.lib.wab_policy_population_grad_stride(env._h, A))
        dev, lib = env.device, self.lib
        lin = int(lib.wab_policy_linear_packed_bytes(150, 128))
        if lin != int(lib.wab_policy_linear_packed_bytes(128, 150)):
            raise RuntimeError("the stacked layouts assume one packed size for every trunk layer")
        u8 = dict(dtype=torch.uint8, device=dev)
        self.packed1 = torch.empty(P, int(lib.wab_policy_affine1_packed_bytes()), **u8)
        self.packed2, self.packed3, self.packed2t, self.packed3t = (torch.empty(P, lin, **u8) for _ in range(4))
        self.bias1, self.bias2, self.bias3 = (torch.empty(P, k, device=dev) for k in (128, 150, 128))
        self.w_heads, self.b_heads = torch.empty(P, A + 1, 128, device=dev), torch.empty(P, A + 1, device=dev)
        self.scratch = torch.empty(int(lib.wab_policy_backward_population_scratch_bytes(env._h, P)), **u8)
        self._packed_versions = [None] * P
        self.refresh()

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream)

    def _versions(self, p: int) -> tuple:
        return tuple((id(prm), prm._version) for prm in self.policies[p].parameters())

    @torch.no_grad()
    def refresh(self, members=None):
        """Re-pack members ``members`` (default: all) into their rows of the stacked buffers."""
        lib, s = self.lib, self._stream()
        f = lambda t: t.detach().float().contiguous()
        for p in range(self.n_members) if members is None else members:
            pol = self.policies[p]
            _lib.check(lib.wab_policy_affine1_prepare(_ptr(f(pol.affine1.weight)), self.env.flat_dim, _ptr(self.packed1[p]), s))
            _lib.check(lib.wab_policy_linear_prepare(_ptr(f(pol.affine2.weight)), 150, 128, _ptr(self.packed2[p]), s))
            _lib.check(lib.wab_policy_linear_prepare(_ptr(f(pol.affine3.weight)), 128, 150, _ptr(self.packed3[p]), s))
            _lib.check(lib.wab_policy_linear_prepare(_ptr(f(pol.affine2.weight.t())), 128, 150, _ptr(self.packed2t[p]), s))
            _lib.check(lib.wab_policy_linear_prepare(_ptr(f(pol.affine3.weight.t())), 150, 128, _ptr(self.packed3t[p]), s))
            self.bias1[p].copy_(pol.affine1.bias); self.bias2[p].copy_(pol.affine2.bias); self.bias3[p].copy_(pol.affine3.bias)
            w, b = stacked_heads(pol)
            self.w_heads[p].copy_(w); self.b_heads[p].copy_(b)
            self._packed_versions[p] = self._versions(p)

    def _refresh_stale(self):
        stale = [p for p in range(self.n_members) if self._packed_versions[p] != self._versions(p)]
        if stale:
            self.refresh(stale)

    def forward_sample(self, features: torch.Tensor, actions: torch.Tensor, value: Optional[torch.Tensor] = None,
                       probs: Optional[torch.Tensor] = None, logp: Optional[torch.Tensor] = None, noise_scale: float = 0.01,
                       counter: Optional[torch.Tensor] = None, seed: int = 0, z3: Optional[torch.Tensor] = None,
                       slope: float = 0.01) -> torch.Tensor:
        """``PolicyTrunkTC.forward_sample`` for the N = P n rows of ``features`` u8[N, 28], row r under member r // n's
        weights, in ONE launch. Fills ``actions`` u8[N] (and ``value`` f32[N], ``probs`` f32[N, A], ``logp`` f32[N],
        ``z3`` f32[N, 128] when given)."""
        self._check_forward(features, actions, value, probs, logp, z3, counter)
        return self._launch(int(seed), features, actions, value, probs, logp, z3, noise_scale, counter, slope)

    def forward_greedy(self, features: torch.Tensor, actions: torch.Tensor, value: Optional[torch.Tensor] = None,
                       probs: Optional[torch.Tensor] = None, logp: Optional[torch.Tensor] = None, noise_scale: float = 0.01,
                       counter: Optional[torch.Tensor] = None, z3: Optional[torch.Tensor] = None,
                       slope: float = 0.01) -> torch.Tensor:
        """``PolicyTrunkTC.forward_greedy`` for every member in ONE launch (``wab_policy_act_population``): row r's action is
        the argmax of member r // n's logits; the arguments and their checks are ``forward_sample``'s, without a seed."""
        self._check_forward(features, actions, value, probs, logp, z3, counter)
        return self._launch(None, features, actions, value, probs, logp, z3, noise_scale, counter, slope)

    def _launch(self, seed, features, actions, value, probs, logp, z3, noise_scale, counter, slope):
        """The launch of ``forward_sample`` (``seed`` given) or ``forward_greedy`` (``seed`` None) without the checks and
        the re-pack: for a caller that checked its own buffers and packed its members once (``PopulationEvaluator``)."""
        common = (self.env._h, _ptr(features), self.n_members, self.member_envs, _ptr(self.packed1), _ptr(self.bias1),
                  _ptr(self.packed2), _ptr(self.bias2), 150, _ptr(self.packed3), _ptr(self.bias3), _ptr(self.w_heads),
                  _ptr(self.b_heads), self.n_actions, float(noise_scale), float(slope), -4.0, 4.0)
        outs = (_ptr(counter), _ptr(actions), _ptr(value), _ptr(probs), _ptr(logp), _ptr(z3), self._stream())
        if seed is None:
            _lib.check(self.lib.wab_policy_act_population(*common, *outs))
        else:
            _lib.check(self.lib.wab_policy_forward_population(*common, seed & (2 ** 64 - 1), *outs))
        return actions

    def _check_forward(self, features, actions, value, probs, logp, z3, counter):
        """The argument checks of the forward calls, then a re-pack of the members whose weights changed."""
        N, A = self.n_members * self.member_envs, self.n_actions
        if tuple(features.shape) != (N, 28) or features.dtype != torch.uint8 or not features.is_contiguous():
            raise ValueError("features must be a contiguous uint8 [P n, 28] tensor")
        if tuple(actions.shape) != (N,) or actions.dtype != torch.uint8 or not actions.is_contiguous():
            raise ValueError("actions must be a contiguous uint8 [P n] tensor")
        for name, t, shape in (("value", value, (N,)), ("probs", probs, (N, A)), ("logp", logp, (N,)), ("z3", z3, (N, 128))):
            if t is not None and (t.dtype != torch.float32 or tuple(t.shape) != shape or not t.is_contiguous()):
                raise ValueError("%s must be a contiguous float32 %s tensor" % (name, list(shape)))
        for name, t in (("features", features), ("actions", actions), ("value", value), ("probs", probs), ("logp", logp),
                        ("z3", z3), ("counter", counter)):
            if t is not None and t.device != self.env.device:
                raise ValueError("%s must be on the environment's device" % name)
        self._refresh_stale()

    def ppo_backward(self, features: torch.Tensor, counters: torch.Tensor, actions: torch.Tensor, logp_old: torch.Tensor,
                     advantage: torch.Tensor, target: torch.Tensor, rows: torch.Tensor, counts: torch.Tensor, coefs,
                     out: Optional[torch.Tensor] = None, logp: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None,
                     entropy: Optional[torch.Tensor] = None, noise_scale: float = 0.01, slope: float = 0.01) -> torch.Tensor:
        """``PolicyTrainTC.ppo_backward`` for every member in ONE launch. ``rows`` int32[P, M]: member p's row list as
        GLOBAL rows t N + n (an entry outside [0, T N) or in another member's block contributes nothing); ``counts``
        int64[P] on the device: member p uses its first ``counts[p]`` entries. ``coefs``: P rows of (clip_eps,
        policy_weight, value_weight, entropy_weight) on the host. Returns ``out`` f32[P, grad_stride]: row p's first
        ``n_params`` floats are member p's flat gradient. ``logp``, ``value``, ``entropy`` f32[T, N] as for one policy."""
        T, N = actions.shape
        P = self.n_members
        if N != P * self.member_envs:
            raise ValueError("actions must be [T, P n]")
        if tuple(features.shape) != (T, N, 28) or features.dtype != torch.uint8 or not features.is_contiguous():
            raise ValueError("features must be a contiguous uint8 [T, N, 28] tensor")
        for name, t in (("logp_old", logp_old), ("advantage", advantage), ("target", target)):
            if t.dtype != torch.float32 or tuple(t.shape) != (T, N) or not t.is_contiguous():
                raise ValueError("%s must be a contiguous float32 [T, N] tensor" % name)
        for name, t in (("logp", logp), ("value", value), ("entropy", entropy)):
            if t is not None and (t.dtype != torch.float32 or tuple(t.shape) != (T, N) or not t.is_contiguous()):
                raise ValueError("%s must be a contiguous float32 [T, N] tensor" % name)
        if counters.dtype != torch.int64 or counters.numel() != T or actions.dtype != torch.uint8 or not actions.is_contiguous():
            raise ValueError("counters must be int64[T], actions a contiguous uint8 [T, N] tensor")
        if rows.dtype != torch.int32 or rows.dim() != 2 or rows.shape[0] != P or not rows.is_contiguous():
            raise ValueError("rows must be a contiguous int32 [P, M] tensor")
        if counts.dtype != torch.int64 or tuple(counts.shape) != (P,) or not counts.is_contiguous():
            raise ValueError("counts must be a contiguous int64 [P] tensor")
        if len(coefs) != P or any(len(row) != 4 for row in coefs):
            raise ValueError("coefs must hold P rows of (clip_eps, policy_weight, value_weight, entropy_weight)")
        coef = (ctypes.c_float * (4 * P))(*(float(c) for row in coefs for c in row))
        if out is None:
            out = torch.empty(P, self.grad_stride, dtype=torch.float32, device=self.env.device)
        if out.dtype != torch.float32 or tuple(out.shape) != (P, self.grad_stride) or not out.is_contiguous():
            raise ValueError("out must be a contiguous float32 [P, grad_stride] tensor")
        for name, t in (("features", features), ("counters", counters), ("actions", actions), ("logp_old", logp_old),
                        ("advantage", advantage), ("target", target), ("rows", rows), ("counts", counts), ("out", out),
                        ("logp", logp), ("value", value), ("entropy", entropy)):
            if t is not None and t.device != self.env.device:
                raise ValueError("%s must be on the environment's device" % name)
        self._refresh_stale()
        _lib.check(self.lib.wab_policy_ppo_backward_population(
            self.env._h, _ptr(features), T, N, P, _ptr(counters), _ptr(actions), _ptr(logp_old), _ptr(advantage),
            _ptr(target), _ptr(rows), rows.shape[1], _ptr(counts), _ptr(self.packed1), _ptr(self.bias1), _ptr(self.packed2),
            _ptr(self.bias2), 150, _ptr(self.packed3), _ptr(self.bias3), _ptr(self.packed2t), _ptr(self.packed3t),
            _ptr(self.w_heads), _ptr(self.b_heads), self.n_actions, float(noise_scale), float(slope), -4.0, 4.0,
            ctypes.cast(coef, ctypes.c_void_p), _ptr(self.scratch), self.scratch.numel(), _ptr(out), _ptr(logp), _ptr(value),
            _ptr(entropy), self._stream()))
        return out

    def grad_f64(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The gradient of the last ``ppo_backward`` on this stream as f64[P, grad_stride]: every member's fixed-order fp64
        sum over its CTAs, not rounded, padding 0 (``wab_policy_backward_population_grad_f64``). For a cross-rank sum that
        rounds once."""
        shape = (self.n_members, self.grad_stride)
        if out is None:
            out = torch.empty(shape, dtype=torch.float64, device=self.env.device)
        if out.dtype != torch.float64 or tuple(out.shape) != shape or not out.is_contiguous() or out.device != self.env.device:
            raise ValueError("out must be a contiguous float64 [P, grad_stride] tensor on the environment's device")
        _lib.check(self.lib.wab_policy_backward_population_grad_f64(self.env._h, _ptr(self.scratch), self.scratch.numel(),
                                                                    self.n_members, self.n_actions, _ptr(out), self._stream()))
        return out

    def grad_sum_ranks(self, rank_grads: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """fp32 of the fp64 sum over ranks, in rank order, of ``rank_grads`` f64[W, P, grad_stride] into ``out`` f32[P,
        grad_stride] (``wab_policy_grad_sum_ranks`` over P grad_stride elements)."""
        shape = (self.n_members, self.grad_stride)
        if rank_grads.dtype != torch.float64 or rank_grads.dim() != 3 or tuple(rank_grads.shape[1:]) != shape or \
                not rank_grads.is_contiguous() or rank_grads.device != self.env.device:
            raise ValueError("rank_grads must be a contiguous float64 [W, P, grad_stride] tensor on the environment's device")
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.env.device)
        if out.dtype != torch.float32 or tuple(out.shape) != shape or not out.is_contiguous() or out.device != self.env.device:
            raise ValueError("out must be a contiguous float32 [P, grad_stride] tensor on the environment's device")
        _lib.check(self.lib.wab_policy_grad_sum_ranks(_ptr(rank_grads), rank_grads.shape[0], out.numel(), _ptr(out),
                                                      self._stream()))
        return out


class _LogitsAndValue(torch.autograd.Function):
    """``PolicyTrainTC.logits_and_value``: forward ``wab_policy_evaluate``, backward ``wab_policy_backward_logits`` into a
    fresh flat gradient per call (a buffer reused across calls would alias an accumulated ``.grad``), returned as views in
    ``parameters_to_vector`` order. The parameters are inputs, saved with the recorded rows, so that autograd checks their
    versions."""

    @staticmethod
    def forward(ctx, tc, features, counters, rows, noise_scale, slope, *params):
        T, N = features.shape[:2]
        M = T * N if rows is None else rows.numel()
        w, b = tc.heads
        A = w.shape[0] - 1
        logits = torch.empty(M, A, dtype=torch.float32, device=features.device)
        value = torch.empty(M, dtype=torch.float32, device=features.device)
        if M > 0:
            _lib.check(tc.lib.wab_policy_evaluate(
                tc.env._h, _ptr(features), T, N, _ptr(counters), _ptr(rows), M, _ptr(tc.packed), _ptr(tc.bias),
                _ptr(tc.packed2), _ptr(tc.bias2), 150, _ptr(tc.packed3), _ptr(tc.bias3), _ptr(w), _ptr(b), A,
                noise_scale, slope, -4.0, 4.0, _ptr(tc.scratch), tc.scratch.numel(), _ptr(logits), _ptr(value), tc._stream()))
        ctx.save_for_backward(features, counters, rows, *params)
        ctx.tc, ctx.noise_scale, ctx.slope, ctx.n_rows = tc, noise_scale, slope, M
        return logits, value

    @staticmethod
    @once_differentiable
    def backward(ctx, g_logits, g_value):
        features, counters, rows, *params = ctx.saved_tensors      # raises if a parameter changed in place since the forward
        tc, M = ctx.tc, ctx.n_rows
        T, N = features.shape[:2]
        grad = torch.zeros(tc.n_params, dtype=torch.float32, device=features.device) if M == 0 else \
            torch.empty(tc.n_params, dtype=torch.float32, device=features.device)
        if M > 0:
            g_logits = g_logits.float().contiguous()
            g_value = g_value.float().contiguous()
            w, b = tc.heads
            _lib.check(tc.lib.wab_policy_backward_logits(
                tc.env._h, _ptr(features), T, N, _ptr(counters), _ptr(rows), M, _ptr(g_logits), _ptr(g_value),
                _ptr(tc.packed), _ptr(tc.bias), _ptr(tc.packed2), _ptr(tc.bias2), 150, _ptr(tc.packed3), _ptr(tc.bias3),
                _ptr(tc.packed2t), _ptr(tc.packed3t), _ptr(w), _ptr(b), w.shape[0] - 1, ctx.noise_scale, ctx.slope, -4.0, 4.0,
                _ptr(tc.scratch), tc.scratch.numel(), _ptr(grad), tc._stream()))
        out, off = [], 0
        for i, p in enumerate(params):
            out.append(grad[off:off + p.numel()].view_as(p) if ctx.needs_input_grad[6 + i] else None)
            off += p.numel()
        return (None, None, None, None, None, None, *out)


class Rollout:
    """N-environment rollout with every tensor resident on the device.

    ``step()`` = flatten features -> + U[0,1)/100 noise -> policy -> Categorical sample -> env.step.
    With ``use_graph=True`` one step is captured in a CUDA graph and replayed (the loop is launch-bound
    for small batches)."""

    def __init__(self, env: VecEnv, policy: Optional[Policy] = None, noise: bool = True, use_graph: bool = False,
                 dtype: torch.dtype = torch.float32, fused_tail: Optional[bool] = None, track_reward: bool = False,
                 tc_first_layer: Optional[bool] = None, tc_trunk: Optional[bool] = None):
        if not env.with_features:
            raise ValueError("Rollout needs VecEnv(features=True)")
        self.env, self.noise, self.dtype = env, noise, dtype
        self.policy = (policy or Policy(env.flat_dim, env.n_actions)).to(env.device).to(dtype).eval()
        self.flat = torch.empty(env.num_envs, env.flat_dim, dtype=dtype, device=env.device)   # policy input, its dtype
        self.noise_ctr = torch.zeros(1, dtype=torch.int64, device=env.device)                  # draw counter (graph-safe)
        self.sample_seed = int(torch.initial_seed()) & (2 ** 63 - 1)
        self.actions = torch.zeros(env.num_envs, dtype=torch.uint8, device=env.device)
        self.values = torch.zeros(env.num_envs, dtype=torch.float32, device=env.device)
        self.reward_sum = torch.zeros((), dtype=torch.float64, device=env.device)
        self.track_reward = track_reward         # episode statistics live in env.stats(); summing rewards here is optional
        # fp32: the trunk's three GEMMs stay library calls (cuBLAS), everything after affine3 is one kernel of this library
        self.fused_tail = (dtype == torch.float32) if fused_tail is None else bool(fused_tail)
        if self.fused_tail and dtype != torch.float32:
            raise ValueError("the fused policy tail is an fp32 kernel")
        self.heads = stacked_heads(self.policy) if self.fused_tail else None
        # fp32: the first layer (input generation + 449 x 128 product + activation) is one tcgen05 kernel of this library
        self.tc_first_layer = self.fused_tail if tc_first_layer is None else bool(tc_first_layer)
        if self.tc_first_layer and not self.fused_tail:
            raise ValueError("the tensor-core first layer belongs to the fp32 fused path")
        # ... and so is the whole trunk (the default): features -> z3 without the hidden activations leaving the SM
        self.tc_trunk = self.tc_first_layer if tc_trunk is None else bool(tc_trunk)
        if self.tc_trunk and not self.tc_first_layer:
            raise ValueError("the tensor-core trunk includes the tensor-core first layer")
        self.affine1_tc = (PolicyTrunkTC if self.tc_trunk else Affine1TC)(env, self.policy) if self.tc_first_layer else None
        self.h1 = torch.empty(env.num_envs, 128, dtype=torch.float32, device=env.device) if self.tc_first_layer else None
        env.reset()
        self.graph = None
        if use_graph:
            self._capture(warmup=3)

    def _capture(self, warmup: int):
        env = self.env
        side = torch.cuda.Stream(device=env.device)
        side.wait_stream(torch.cuda.current_stream(env.device))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._step_eager()
            side.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=side):
                self._step_eager()
        torch.cuda.current_stream(env.device).wait_stream(side)

    @torch.no_grad()
    def _step_eager(self):
        env = self.env
        if self.tc_trunk:
            # Policy.forward + select_action (actor_critic.py:84-97, :108-125, :188-189) in one tcgen05 kernel
            self.noise_ctr += 1
            self.affine1_tc.forward_sample(env.last_features, self.heads, self.actions, value=self.values,
                                           noise_scale=0.01 if self.noise else 0.0, counter=self.noise_ctr, seed=self.sample_seed)
            _, reward, _, _ = env.step(self.actions)
            if self.track_reward:
                self.reward_sum += reward.sum(dtype=torch.float64)
            return
        if self.tc_first_layer:
            # flatten (actor_critic.py:188) + U[0,1)/100 noise (:189) + affine1 + leaky_relu (:88-90): one tcgen05 kernel
            h = self.affine1_tc(env.last_features, self.h1, 0.01 if self.noise else 0.0, self.noise_ctr)
        else:
            # gym.spaces.flatten (actor_critic.py:188) + U[0,1)/100 input noise (:189) + cast, one kernel
            env.flatten_features_noisy(env.last_features, self.flat, 0.01 if self.noise else 0.0, self.noise_ctr)
        self.noise_ctr += 1
        if self.fused_tail:
            p = self.policy
            if not self.tc_first_layer:
                h = F.leaky_relu(p.affine1(self.flat))                                   # :88-90 (cuBLAS)
            z3 = h if self.tc_trunk else p.affine3(F.leaky_relu(p.affine2(h)))           # the trunk kernel already returned z3
            policy_tail(p, z3, self.heads, self.actions, value=self.values, counter=self.noise_ctr, seed=self.sample_seed)
        else:
            probs, value = self.policy(self.flat)
            env.sample_actions(probs, self.actions, self.noise_ctr, seed=self.sample_seed)   # Categorical(probs).sample(), :117-120
            self.values.copy_(value.squeeze(1))
        _, reward, _, _ = env.step(self.actions)
        if self.track_reward:
            self.reward_sum += reward.sum(dtype=torch.float64)

    def describe(self) -> str:
        if self.tc_trunk:
            return ("wab_affine1_tc_kernel<2> (ONE tcgen05 kernel: flatten + noise + affine1..3 + leaky_relu with bf16 x 3 splits and fp32 "
                    "accumulation, activations stay on the SM; then clamp, both heads, softmax, Categorical sample) -> wab_step_kernel; "
                    "one CUDA graph per step")
        if self.tc_first_layer:
            return ("wab_affine1_tc_kernel (flatten + noise + affine1 + leaky_relu: tcgen05, bf16 x 3 splits, fp32 accumulate) -> "
                    "affine2, affine3 fp32 (cuBLAS) + leaky_relu -> wab_policy_tail_kernel (activation, clamp, both heads, softmax, "
                    "Categorical sample) -> wab_step_kernel; one CUDA graph per step")
        if self.fused_tail:
            return ("wab_flatten_noisy_kernel (flatten + noise) -> affine1..3 fp32 (cuBLAS) + leaky_relu -> wab_policy_tail_kernel "
                    "(activation, clamp, both heads, softmax, Categorical sample) -> wab_step_kernel; one CUDA graph per step")
        return "wab_flatten_noisy_kernel -> torch MLP (cuBLAS) -> wab_sample_kernel -> wab_step_kernel; one CUDA graph per step"

    def refresh_weights(self):
        """After an optimiser step: re-pack what the kernels hold of the policy (stacked heads, split tensor-core operands).
        The buffers are updated in place, so a captured graph keeps working."""
        if self.heads is not None:
            w, b = stacked_heads(self.policy)
            self.heads[0].copy_(w); self.heads[1].copy_(b)
        if self.affine1_tc is not None:
            self.affine1_tc.refresh()

    def state_dict(self) -> dict:
        """Environment state (``VecEnv.state_dict``), policy weights, the noise / sampling draw counter and the sampling seed:
        a rollout resumed from it produces the same actions, values and rewards as one that never stopped."""
        return {"env": self.env.state_dict(), "policy": {k: v.detach().cpu().clone() for k, v in self.policy.state_dict().items()},
                "noise_ctr": int(self.noise_ctr.item()), "sample_seed": self.sample_seed}

    def load_state_dict(self, sd: dict):
        """Resume from ``state_dict()``. Every tensor is loaded in place, so a captured CUDA graph keeps working; a
        different sampling seed (a kernel argument of the graph) is captured anew, without stepping."""
        self.env.load_state_dict(sd["env"])
        self.policy.load_state_dict(sd["policy"])
        self.refresh_weights()
        self.noise_ctr.fill_(int(sd["noise_ctr"]))
        if int(sd["sample_seed"]) != self.sample_seed:
            self.sample_seed = int(sd["sample_seed"])
            if self.graph is not None:
                self._capture(warmup=0)

    def step(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self._step_eager()

    def run(self, steps: int) -> Dict[str, float]:
        for _ in range(steps):
            self.step()
        return {"env_steps": steps * self.env.num_envs}
