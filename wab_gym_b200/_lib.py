"""ctypes binding of ``libwab_b200.so`` (the C ABI of ``include/wab_b200.h``).

There is deliberately no fallback: if the library cannot be built or loaded, importing a VecEnv
fails loudly. Nothing here (or anywhere in this package) imports ``oracle/``.
"""
import ctypes
import os
import shutil
import warnings

from . import build as _build
from .config import WabConfigStruct

_lib = None

EXPORTS = [
    "wab_vec_create", "wab_vec_reset", "wab_vec_step", "wab_vec_step_many", "wab_vec_step_host",
    "wab_vec_reset_host", "wab_vec_stats", "wab_vec_stats_device", "wab_vec_export_state", "wab_vec_num_envs", "wab_vec_lanes_per_env", "wab_vec_step_many_pipelined", "wab_vec_kernel_kind",
    "wab_vec_destroy", "wab_philox_device", "wab_vec_bind_features", "wab_pragmatic_features",
    "wab_vec_flatten_features", "wab_vec_flatten_features_noisy", "wab_sample_categorical", "wab_policy_tail", "wab_vec_enable_ego", "wab_vec_set_replicas", "wab_vec_set_blocks", "wab_vec_ego_proximities", "wab_vec_flat_dim", "wab_vec_host_block_layout", "wab_vec_step_host_packed", "wab_vec_forget_host_buffers",
    "wab_vec_state_record_bytes", "wab_vec_state_fingerprint", "wab_vec_save_state", "wab_vec_load_state", "wab_vec_set_stats",
    "wab_policy_affine1_packed_bytes", "wab_policy_affine1_prepare", "wab_policy_affine1", "wab_policy_linear_packed_bytes", "wab_policy_linear_prepare", "wab_policy_trunk", "wab_policy_forward", "wab_policy_act", "wab_policy_backward_scratch_bytes", "wab_policy_backward", "wab_policy_ppo_backward", "wab_policy_evaluate", "wab_policy_backward_logits", "wab_policy_backward_grad_f64", "wab_policy_grad_sum_ranks", "wab_policy_backward_population_grad_f64", "wab_policy_forward_population", "wab_policy_act_population", "wab_policy_backward_population_scratch_bytes", "wab_policy_population_grad_stride", "wab_policy_ppo_backward_population", "wab2_create", "wab2_kernel_kind", "wab2_output_layout", "wab2_reset", "wab2_turn", "wab2_export_state", "wab2_import_state", "wab2_destroy", "wab_last_error", "wab_abi_version",
]


class WabObs(ctypes.Structure):
    _fields_ = [("d_grids", ctypes.c_void_p), ("d_food", ctypes.c_void_p), ("d_role", ctypes.c_void_p),
                ("d_status", ctypes.c_void_p)]


class WabError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("wab_b200 error %d: %s" % (code, message))
        self.code = code


def load():
    """Load (building first if stale) the CUDA library. Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("WAB_LIB") or _build.LIB_PATH   # WAB_LIB: a differently-tuned build (tools/tune.py)
    if path == _build.LIB_PATH and _build.is_stale():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this box: only acceptable if a prebuilt library travelled here
            if not os.path.exists(path):
                raise ImportError("libwab_b200.so is missing and could not be built: %s" % exc) from exc
            if shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc"):
                raise ImportError("libwab_b200.so is older than its sources and the rebuild failed: %s" % exc) from exc
            warnings.warn("libwab_b200.so is older than its sources and there is no nvcc here to rebuild it; "
                          "loading the prebuilt library")
    L = ctypes.CDLL(path)
    vp, i32, i64, u64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64
    L.wab_vec_create.argtypes = [ctypes.POINTER(WabConfigStruct), vp, i32, i64, u64, u64, i32, ctypes.POINTER(vp)]
    L.wab_vec_reset.argtypes = [vp, vp, WabObs, vp]
    L.wab_vec_step.argtypes = [vp, vp, WabObs, vp, vp, vp, vp]
    L.wab_vec_step_many.argtypes = [vp, i32, vp, WabObs, vp, vp, vp, vp]
    L.wab_vec_step_host.argtypes = [vp] * 10
    L.wab_vec_reset_host.argtypes = [vp] * 6
    L.wab_vec_host_block_layout.argtypes = [vp, vp, vp]
    L.wab_vec_step_host_packed.argtypes = [vp, vp, vp, vp]
    L.wab_vec_forget_host_buffers.argtypes = [vp]
    L.wab_vec_stats.argtypes = [vp, vp, i32, vp]
    L.wab_vec_stats_device.argtypes = [vp, vp, vp]
    L.wab_vec_export_state.argtypes = [vp] * 14
    L.wab_vec_state_record_bytes.argtypes = [vp]
    L.wab_vec_state_record_bytes.restype = i64
    L.wab_vec_state_fingerprint.argtypes = [vp, vp]
    L.wab_vec_save_state.argtypes = [vp, vp, i64, vp, vp]
    L.wab_vec_load_state.argtypes = [vp, vp, vp, i64, WabObs, vp, vp]
    L.wab_vec_set_stats.argtypes = [vp, vp, vp]
    L.wab_vec_num_envs.argtypes = [vp]
    L.wab_vec_num_envs.restype = i64
    L.wab_vec_kernel_kind.argtypes = [vp]
    L.wab_vec_lanes_per_env.argtypes = [vp]
    L.wab_vec_lanes_per_env.restype = i32
    L.wab_vec_step_many_pipelined.argtypes = [vp, i32]
    L.wab_vec_step_many_pipelined.restype = i32
    L.wab_vec_destroy.argtypes = [vp]
    L.wab_vec_destroy.restype = None
    L.wab_vec_bind_features.argtypes = [vp, vp]
    L.wab_pragmatic_features.argtypes = [vp, vp, vp, vp, i64, vp, vp]
    L.wab_vec_flatten_features.argtypes = [vp, vp, i64, vp, vp]
    L.wab_vec_flatten_features_noisy.argtypes = [vp, vp, i64, vp, ctypes.c_int32, ctypes.c_float, vp, vp]
    L.wab_sample_categorical.argtypes = [vp, ctypes.c_int32, i64, ctypes.c_int32, ctypes.c_uint64, vp, vp, vp]
    L.wab_policy_tail.argtypes = [vp, i32, vp, vp, i64, i32, ctypes.c_float, ctypes.c_float, ctypes.c_float, u64, vp, vp, vp, vp, vp, vp]
    L.wab_vec_enable_ego.argtypes = [vp]
    L.wab_vec_set_replicas.argtypes = [vp, i64]
    L.wab_vec_set_blocks.argtypes = [vp, i64, i64]
    L.wab_vec_ego_proximities.argtypes = [vp, vp, vp]
    L.wab_vec_flat_dim.argtypes = [vp]
    L.wab_vec_flat_dim.restype = i32
    L.wab_policy_affine1_packed_bytes.argtypes = []
    L.wab_policy_affine1_packed_bytes.restype = i64
    L.wab_policy_affine1_prepare.argtypes = [vp, i32, vp, vp]
    L.wab_policy_affine1.argtypes = [vp, vp, i64, vp, vp, ctypes.c_float, ctypes.c_float, vp, vp, vp]
    L.wab_policy_linear_packed_bytes.argtypes = [i32, i32]
    L.wab_policy_linear_packed_bytes.restype = i64
    L.wab_policy_linear_prepare.argtypes = [vp, i32, i32, vp, vp]
    L.wab_policy_trunk.argtypes = [vp, vp, i64, vp, vp, vp, vp, i32, vp, vp, ctypes.c_float, ctypes.c_float, vp, vp, vp]
    L.wab_policy_forward.argtypes = [vp, vp, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, ctypes.c_float, ctypes.c_float,
                                     ctypes.c_float, ctypes.c_float, u64, vp, vp, vp, vp, vp, vp, vp]
    L.wab_policy_act.argtypes = [vp, vp, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, ctypes.c_float, ctypes.c_float,
                                 ctypes.c_float, ctypes.c_float, vp, vp, vp, vp, vp, vp, vp]
    L.wab_policy_backward_scratch_bytes.argtypes = [vp]
    L.wab_policy_backward_scratch_bytes.restype = i64
    f32 = ctypes.c_float
    L.wab_policy_backward.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, i32,
                                      f32, f32, f32, f32, vp, i64, vp, vp, vp, vp]
    L.wab_policy_ppo_backward.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp,
                                          vp, i32, f32, f32, f32, f32, f32, f32, f32, f32, vp, i64, vp, vp, vp, vp, vp]
    L.wab_policy_evaluate.argtypes = [vp, vp, i64, i64, vp, vp, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, f32, f32, f32, f32,
                                      vp, i64, vp, vp, vp]
    L.wab_policy_backward_logits.argtypes = [vp, vp, i64, i64, vp, vp, i64, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp,
                                             i32, f32, f32, f32, f32, vp, i64, vp, vp]
    L.wab_policy_backward_grad_f64.argtypes = [vp, vp, i64, i32, vp, vp]
    L.wab_policy_grad_sum_ranks.argtypes = [vp, i32, i64, vp, vp]
    L.wab_policy_backward_population_grad_f64.argtypes = [vp, vp, i64, i32, i32, vp, vp]
    L.wab_policy_forward_population.argtypes = [vp, vp, i32, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, f32, f32, f32, f32, u64,
                                                vp, vp, vp, vp, vp, vp, vp]
    L.wab_policy_act_population.argtypes = [vp, vp, i32, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, f32, f32, f32, f32,
                                            vp, vp, vp, vp, vp, vp, vp]
    L.wab_policy_backward_population_scratch_bytes.argtypes = [vp, i32]
    L.wab_policy_backward_population_scratch_bytes.restype = i64
    L.wab_policy_population_grad_stride.argtypes = [vp, i32]
    L.wab_policy_population_grad_stride.restype = i64
    L.wab_policy_ppo_backward_population.argtypes = [vp, vp, i64, i64, i32, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, i32,
                                                     vp, vp, vp, vp, vp, vp, i32, f32, f32, f32, f32, vp, vp, i64, vp, vp, vp, vp,
                                                     vp]
    L.wab2_create.argtypes = [vp, i64, u64, u64, i32, ctypes.POINTER(vp)]
    L.wab2_reset.argtypes = [vp, vp]
    L.wab2_turn.argtypes = [vp] * 7
    L.wab2_export_state.argtypes = [vp] * 5
    L.wab2_destroy.argtypes = [vp]
    L.wab2_kernel_kind.argtypes = [vp]
    L.wab2_output_layout.argtypes = [vp]
    L.wab2_import_state.argtypes = [vp] * 5
    L.wab2_destroy.restype = None
    L.wab_philox_device.argtypes = [vp, ctypes.c_uint32, ctypes.c_uint32, i64, vp, vp]
    L.wab_last_error.restype = ctypes.c_char_p
    L.wab_abi_version.restype = i32
    for name in EXPORTS:
        if name not in ("wab_vec_num_envs", "wab_vec_state_record_bytes", "wab_policy_backward_scratch_bytes", "wab_policy_backward_population_scratch_bytes",
                        "wab_policy_population_grad_stride", "wab_vec_lanes_per_env", "wab_vec_step_many_pipelined", "wab_vec_kernel_kind", "wab_vec_flat_dim", "wab_vec_destroy", "wab2_destroy",
                        "wab_last_error", "wab_abi_version"):
            getattr(L, name).restype = ctypes.c_int
    _lib = L
    return L


def check(rc):
    if rc != 0:
        msg = load().wab_last_error().decode("utf-8", "replace")
        if rc in (2,):  # WAB_E_CONFIG mirrors the reference's ValueError (wab_env.py:147-148)
            raise ValueError(msg)
        if rc == 3:
            raise NotImplementedError(msg)
        raise WabError(rc, msg)
