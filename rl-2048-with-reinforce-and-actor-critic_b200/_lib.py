"""ctypes binding of libb2048.so — the only way the Python host reaches the CUDA kernels.

There is deliberately NO fallback: if the shared library is missing or does not export a symbol
declared in include/b2048.h, importing the product fails loudly."""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libb2048.so")

B2048_MAX_LAYERS = 8
NP_RNG_WORDS = 6        # sizeof(b2048_np_rng) / 8: one NumPy PCG64 generator state per board

REWARD = {"sum": 0, "log2": 1}
BONUS = {"off": 0, "raw": 1, "log2": 2}
OBS = {"none": 0, "raw": 1, "log2": 2, "onehot": 3}
ACT = {"buffer": 0, "random_legal": 1, "random_any": 2, "priority": 3}
ACTV = {"Sigmoid": 0, "ReLU": 1}

F_MASK, F_CHANGED, F_DONE, F_TRUNC, F_OVERFLOW = 0x0F, 0x10, 0x20, 0x40, 0x80


class EnvCfg(C.Structure):
    """b2048_env_cfg (include/b2048.h); mirrors Game2048EnvConfig (reference src/env.py:19-40)."""

    _fields_ = [
        ("reward_mode", C.c_int32), ("bonus_mode", C.c_int32), ("obs_mode", C.c_int32),
        ("use_action_mask", C.c_int32), ("max_steps", C.c_int32), ("action_mode", C.c_int32),
        ("auto_reset", C.c_int32), ("action_priority", C.c_int32),
        ("base_reward_scale", C.c_double), ("empty_tile_reward", C.c_double), ("merge_reward", C.c_double),
        ("bonus_scale", C.c_double), ("step_reward", C.c_double), ("endgame_penalty", C.c_double),
        ("invalid_action_penalty", C.c_double), ("obs_log2_scale", C.c_float), ("reserved_f", C.c_float),
    ]


class MlpDesc(C.Structure):
    """b2048_mlp_desc (include/b2048.h); parameters laid out as the reference stores them (src/MLP.py:45-94)."""

    _fields_ = [
        ("n_layers", C.c_int32), ("activation", C.c_int32), ("obs_mode", C.c_int32), ("obs_log2_scale", C.c_float),
        ("dims", C.c_int32 * (B2048_MAX_LAYERS + 1)),
        ("W", C.c_void_p * B2048_MAX_LAYERS), ("b", C.c_void_p * B2048_MAX_LAYERS),
    ]


DEBUG_OPTIONS = {"no_fused_rollout": 0, "no_fast_step": 1, "tc_clocks": 2, "step_clocks": 3, "no_pdl": 4, "no_update_pipe": 5,
                 "pipe_split": 16}


class B2048Error(RuntimeError):
    pass


_vp, _i64, _u64, _u32, _i32, _f32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_uint32, C.c_int32, C.c_float

# symbol -> argtypes; every symbol of include/b2048.h must be here (tests/test_abi.py checks both ways)
SIGNATURES = {
    "b2048_create": [C.POINTER(_vp)],
    "b2048_destroy": [_vp],
    "b2048_version": [],
    "b2048_debug_set": [_vp, _i32, _i32],
    "b2048_get_row_lut": [_vp, _vp, _vp],
    "b2048_reset_many": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _u64, _u64, _u32, _vp],
    "b2048_step_many": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(EnvCfg), _vp, _vp, _vp, _vp, _vp,
                        _vp, _u32, _i64, _u64, _u64, _u32, _vp],
    "b2048_step_many_n": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, C.POINTER(EnvCfg), _vp, _vp, _vp, _i64, _i32, _u64, _u64, _u32, _vp],
    "b2048_move_many": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    "b2048_encode_obs": [_vp, _vp, _i32, _f32, _i64, _vp],
    "b2048_symmetries": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp],
    "b2048_policy_step": [_vp, _vp, _vp, C.POINTER(MlpDesc), _vp, _vp, _vp, _i64, _u64, _u64, _u32, _i32, _i32, _vp],
    "b2048_rollout_many": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(EnvCfg), C.POINTER(MlpDesc), _i64, _i32, _i32,
                           _u64, _u64, _u32, _i32, _i32, _i32, _vp, _i64, _vp, _vp],
    "b2048_compact_live": [_vp, _vp, _i64, _vp, _vp, _vp],
    "b2048_np_rng_seed": [_vp, _vp, _i64, _vp],
    "b2048_reset_many_np": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    "b2048_rollout_many_np": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(EnvCfg), C.POINTER(MlpDesc), _i64, _i32,
                              _i32, _vp, _vp, _i32, _i32, _vp, _i64, _vp, _vp],
    "b2048_mlp_forward": [_vp, _vp, C.POINTER(MlpDesc), _vp, _i64, _i32, _vp],
    "b2048_dense_forward": [_vp, _vp, C.POINTER(MlpDesc), _vp, _vp, _i64, _vp],
    "b2048_reverse_scan": [_vp, _vp, _vp, _f32, _i32, _i64, _vp],
    "b2048_reverse_scan_f64": [_vp, _vp, _vp, C.c_double, _i32, _i64, _vp],
    "b2048_advantages": [_vp, _vp, _vp, _vp, _i32, _f32, _i32, _i64, _vp, _vp, _vp, _i32, _vp, _vp],
    "b2048_weighted_stats": [_vp, _vp, _vp, _vp, _i32, _i64, _vp, _vp],
    "b2048_td_errors": [_vp, _vp, _vp, _vp, _vp, _f32, _i32, _f32, _f32, _i32, _i64, _vp, _vp, _vp],
    "b2048_segment_targets": [_vp, _vp, _vp, _vp, C.c_double, C.c_double, _i32, _f32, _f32, _i32, _i64, _vp, _vp, _vp, _vp,
                              _vp],
    "b2048_advantages_window": [_vp, _vp, _vp, _i32, _f32, _i32, _i64, _vp, _vp, _vp, _i32, _vp],
    "b2048_horizon_episodes": [_vp, _vp, _vp, _vp, _vp, _i32, _i64, _vp, _vp, _vp],
    "b2048_replay_pre_reset": [_vp, _vp, _vp, _vp, _i64, _i64, _u64, _u64, _u32, _vp, _vp],
    "b2048_fold_bootstrap": [_vp, _vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp],
    "b2048_ppo_minibatches": [_vp, _i32, _i64, _i64, _i64, _i64, _u64, _u32, _vp, _vp],
    "b2048_ppo_logp": [_vp, _vp, _vp, _vp, _i64, _vp, _vp],
    "b2048_ppo_coefficients": [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_double, C.c_double, C.c_double, _i32,
                               _f32, _vp, _vp, _vp, _vp],
    "b2048_lookahead_expand": [_vp, _vp, _vp, _vp, C.POINTER(EnvCfg), _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp,
                               _vp],
    "b2048_lookahead_select": [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _vp],
    "b2048_backward_workspace_floats": [C.POINTER(MlpDesc), _i64],
    "b2048_mlp_backward": [_vp, _vp, _vp, _vp, _vp, C.POINTER(MlpDesc), _vp, _i64, _i32, _vp, _i64, _i64, _i32, _vp],
    "b2048_mlp_backward_entropy": [_vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(MlpDesc), _vp, _i64, _vp, _i64, _i64, _i32, _vp,
                                   _vp],
    "b2048_backward_tc_layout": [_i64, _vp],
    "b2048_apply_update": [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _f32, _f32, _f32, _f32, _f32, _i32, _vp, _vp],
}

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B2048Error(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    import torch  # noqa: F401  (libb2048 links the shared CUDA runtime; torch has already mapped libcudart.so.12)
    lib = C.CDLL(LIB_PATH)
    lib.b2048_last_error.restype = C.c_char_p
    lib.b2048_last_error.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI mismatch, on purpose
        fn.argtypes = argtypes
        fn.restype = C.c_int64 if name == "b2048_backward_workspace_floats" else C.c_int
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().b2048_last_error()
        raise B2048Error(f"{what} failed with status {status}: {msg.decode() if msg else ''}")
