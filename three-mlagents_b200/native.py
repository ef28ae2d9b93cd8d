"""ctypes binding of libtmla.so (include/tmla.h) — the only way into the CUDA hot path.

There is deliberately no fallback: if the library is missing or cannot be loaded, importing this
module raises, and every op that needs it fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TMLA_LIB selects another build of the same library (A/B runs of kernel variants: profiles/train_variants.py)
LIB_PATH = os.environ.get("TMLA_LIB") or os.path.join(_HERE, "lib", "libtmla.so")

TMLA_OK, TMLA_EINVAL, TMLA_ECUDA, TMLA_ENOMEM, TMLA_EACTION = 0, -1, -2, -3, -4
TASK_IDS = {"basic": 0, "ball3d": 1, "gridworld": 2, "push": 3, "walljump": 4, "brickbreak": 5, "bicycle": 6, "glider": 7}


class TmlaError(RuntimeError):
    pass


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing. Build it with `python three-mlagents_b200/build.py` "
            "(needs nvcc). three-mlagents_b200 has no CPU fallback."
        )
    return C.CDLL(LIB_PATH)


lib = _load()

vp, i32, i64, u64, f32, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_double
_i = C.c_int

class RolloutArgs(C.Structure):
    """`tmla_rollout_args` of include/tmla.h, field for field."""
    _fields_ = ([(k, C.c_void_p) for k in ("params", "wpack", "act_cache", "obs", "actions", "log_probs", "rewards", "values", "dones",
                                            "last_values", "advantages", "returns", "logits", "trunc_count", "trunc_index", "trunc_obs",
                                            "trunc_values", "ep_stats", "step_counter")]
                + [("gamma", C.c_double), ("gae_lambda", C.c_double)]
                + [(k, C.c_int32) for k in ("obs_dim", "hidden", "n_actions", "n_steps", "deterministic", "trunc_capacity")])


# name -> (restype, argtypes); mirrors include/tmla.h declaration by declaration
SIGNATURES = {
    "tmla_version": (_i, []),
    "tmla_last_error": (C.c_char_p, []),
    "tmla_task_from_name": (_i, [C.c_char_p]),
    "tmla_task_obs_dim": (_i, [_i]),
    "tmla_task_num_actions": (_i, [_i]),
    "tmla_task_max_steps": (_i, [_i]),
    "tmla_task_state_size": (_i, [_i]),
    "tmla_create": (_i, [_i, i64, u64, u64, _i, C.POINTER(vp)]),
    "tmla_destroy": (_i, [vp]),
    "tmla_seed": (_i, [vp, u64]),
    "tmla_num_envs": (i64, [vp]),
    "tmla_step_count": (u64, [vp]),
    "tmla_reset": (_i, [vp, vp, vp]),
    "tmla_step": (_i, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "tmla_step_host": (_i, [vp, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(i64)]),
    "tmla_reset_host": (_i, [vp, vp]),
    "tmla_host_views": (_i, [vp] + [C.POINTER(vp)] * 8),
    "tmla_step_pinned": (_i, [vp, C.POINTER(i64)]),
    "tmla_host_records": (_i, [vp, C.POINTER(vp), C.POINTER(i32)]),
    "tmla_result_block_layout": (_i, [vp, C.POINTER(i64), C.POINTER(i64)]),
    "tmla_result_block_alloc": (_i, [vp, C.POINTER(vp)]),
    "tmla_result_block_free": (_i, [vp]),
    "tmla_step_block": (_i, [vp, vp, C.POINTER(i64)]),
    "tmla_stage_actions": (_i, [vp, vp, _i]),
    "tmla_step_block_begin": (_i, [vp, vp, _i, vp]),
    "tmla_step_block_end": (_i, [vp, vp, C.POINTER(i64)]),
    "tmla_set_episode_log": (_i, [vp, vp, i32, vp]),
    "tmla_get_state": (_i, [vp, vp, vp]),
    "tmla_set_state": (_i, [vp, vp, vp]),
    "tmla_check_actions": (_i, [vp, vp]),
    "tmla_rollout_random": (_i, [vp, _i, vp, vp, vp, vp, vp]),
    "tmla_step_policy": (_i, [vp, vp, _i, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]),
    "tmla_rollout": (_i, [vp, C.POINTER(RolloutArgs), vp]),
    "tmla_advance_steps": (_i, [vp, u64]),
    "tmla_counter_add": (_i, [vp, u64, vp]),
    "tmla_selftest_arith": (_i, [vp, vp]),
    "tmla_bootstrap_add": (_i, [vp, vp, vp, vp, f64, i32, vp]),
    "tmla_gae": (_i, [vp, vp, vp, vp, f64, f64, _i, i64, vp, vp, vp]),
    "tmla_permutation": (_i, [u64, u64, i64, _i, i64, vp, vp]),
    "tmla_mlp_num_params": (i64, [_i, _i, _i]),
    "tmla_mlp_forward": (_i, [vp, _i, _i, _i, vp, vp, i64, vp, vp, vp, vp, vp]),
    "tmla_mlp_backward_scratch": (i64, [_i, _i, _i, i64]),
    "tmla_mlp_backward": (_i, [vp, _i, _i, _i, vp, vp, i64, vp, vp, vp, vp, vp, vp]),
    "tmla_mlp_pack_bf16": (_i, [vp, _i, _i, _i, vp, vp]),
    "tmla_mlp_forward_bf16": (_i, [vp, vp, _i, _i, _i, vp, vp, i64, vp, vp, vp, vp, vp]),
    "tmla_mlp_backward_bf16": (_i, [vp, vp, _i, _i, _i, vp, vp, i64, vp, vp, vp, vp, vp, vp]),
    "tmla_adv_stats": (_i, [vp, vp, i64, vp, vp]),
    "tmla_adv_stats_batched": (_i, [vp, vp, i64, i64, vp, vp]),
    "tmla_ppo_loss": (_i, [vp, vp, vp, vp, vp, vp, vp, i64, i64, _i, vp, _i, f32, f32, f32, vp, vp, vp, vp]),
    "tmla_a2c_loss": (_i, [vp, vp, vp, vp, vp, vp, i64, i64, _i, vp, _i, f32, f32, vp, vp, vp, vp]),
    "tmla_tc_linear": (_i, [_i, vp, vp, vp, vp, vp, i64, vp, vp]),
    "tmla_tc_wgrad": (_i, [vp, vp, vp, i64, vp]),
    "tmla_f32_to_bf16": (_i, [vp, vp, i64, vp]),
    "tmla_tc_debug": (_i, [_i]),
    "tmla_adam_clip": (_i, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, i64, vp, vp]),
    "tmla_adam_clip_zero": (_i, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, i64, vp, _i, vp]),
    "tmla_adam_clip_fused": (_i, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, i64, vp, _i, vp, _i, _i, _i, vp]),
    "tmla_comm_create": (_i, [_i, _i, _i, i64, C.POINTER(vp), vp]),
    "tmla_comm_connect": (_i, [vp, vp]),
    "tmla_comm_destroy": (_i, [vp]),
    "tmla_comm_check": (_i, [vp, vp]),
    "tmla_adam_clip_allreduce": (_i, [vp, vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, i64, vp, _i, vp, _i, _i, _i, vp]),
    "tmla_rmsprop_clip_fused": (_i, [vp, vp, vp, i64, f32, f32, f32, f64, f32, vp, _i, vp, _i, _i, _i, vp]),
    "tmla_rmsprop_clip_allreduce": (_i, [vp, vp, vp, vp, i64, f32, f32, f32, f64, f32, i64, vp, _i, vp, _i, _i, _i, vp]),
    "tmla_ppo_minibatch_supported": (_i, [_i, _i, _i]),
    "tmla_ppo_minibatch_scratch": (i64, [_i, i64]),
    "tmla_ppo_minibatch_bf16": (_i, [vp, vp, _i, _i, _i, vp, vp, i64, i64, vp, vp, vp, vp, vp, _i, f32, f32, f32, vp, vp, vp,
                                     vp, vp, _i, vp]),
    "tmla_a2c_batch_bf16": (_i, [vp, vp, _i, _i, _i, vp, vp, i64, i64, vp, vp, vp, vp, _i, f32, f32, vp, vp, vp, vp, vp, _i, vp]),
    "tmla_tc_wgrad_tiled": (_i, [vp, vp, vp, i64, vp]),
    "tmla_tc_probe": (_i, [vp, vp, vp, _i, vp]),
    "tmla_tc_overlap_probe": (_i, [vp, _i, _i, _i, vp]),
    "tmla_det_scratch_bytes": (i64, [_i, _i, _i, i64]),
    "tmla_adv_stats_det_scratch_bytes": (i64, [i64, i64]),
    "tmla_mlp_backward_bf16_det": (_i, [vp, vp, _i, _i, _i, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp]),
    "tmla_adv_stats_batched_det": (_i, [vp, vp, i64, i64, vp, vp, vp]),
    "tmla_ppo_loss_det": (_i, [vp, vp, vp, vp, vp, vp, vp, i64, i64, _i, vp, _i, f32, f32, f32, vp, vp, vp, vp, vp]),
    "tmla_a2c_loss_det": (_i, [vp, vp, vp, vp, vp, vp, i64, i64, _i, vp, _i, f32, f32, vp, vp, vp, vp, vp]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)      # AttributeError here = header and library out of sync
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return (lib.tmla_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    """Map the C ABI's error codes onto the exceptions the reference raises
    (ValueError for bad input as in registry.py:368-369 / training.py:105-114)."""
    if rc == TMLA_OK:
        return
    msg = last_error()
    if rc == TMLA_EINVAL:
        raise ValueError(msg)
    if rc == TMLA_EACTION:
        raise IndexError(msg)       # the reference's ACTION_DELTAS[action] raises IndexError
    if rc == TMLA_ENOMEM:
        raise MemoryError(msg)
    raise TmlaError(f"libtmla error {rc}: {msg}")


def ptr(t) -> int | None:
    """Device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
