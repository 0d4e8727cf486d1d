"""ctypes binding of ``libts_b200.so`` (the C ABI declared in ``include/ts_b200.h``).

The library is the product: if it cannot be loaded, every device entry point raises -- there is
no CPU fallback (the numpy/C oracle under ``oracle/`` is test infrastructure and is never imported
from here).  torch is used only as plumbing: device memory, the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Any

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libts_b200.so")

TS_F32, TS_F64 = 0, 1
AC_RELU, AC_CATEGORICAL = 1, 2
LOSS_PPO, LOSS_A2C = 0, 1
STATS_STRIDE = 8
GRAD_EXTRA = 4


class ExtensionMissingError(RuntimeError):
    pass


class ActorCriticDesc(C.Structure):
    _fields_ = [
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("hidden", C.c_int32), ("flags", C.c_int32),
        ("a_w1", C.c_int64), ("a_b1", C.c_int64), ("a_w2", C.c_int64), ("a_b2", C.c_int64),
        ("a_w3", C.c_int64), ("a_b3", C.c_int64), ("a_logstd", C.c_int64),
        ("c_w1", C.c_int64), ("c_b1", C.c_int64), ("c_w2", C.c_int64), ("c_b2", C.c_int64),
        ("c_w3", C.c_int64), ("c_b3", C.c_int64),
        ("n_params", C.c_int64),
    ]


class PPOHParams(C.Structure):
    _fields_ = [
        ("eps_clip", C.c_double), ("dual_clip", C.c_double), ("vf_coef", C.c_double),
        ("ent_coef", C.c_double), ("max_grad_norm", C.c_double), ("adv_eps", C.c_double),
        ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("adam_eps", C.c_double),
        ("weight_decay", C.c_double),
        ("value_clip", C.c_int32), ("advantage_normalization", C.c_int32), ("loss_kind", C.c_int32),
    ]


_P = C.c_void_p
_I64 = C.c_int64
_I32 = C.c_int32
_D = C.c_double

# name -> argtypes (restype is int unless noted); mirrors include/ts_b200.h one to one
SIGNATURES: dict[str, list[Any]] = {
    "ts_gae": [_P, _P, C.c_int, _P, _P, _P, _P, C.c_int, _I64, _D, _D, _P, _D, _P, _P, _P, C.c_int, _P, _P],
    "ts_rms_merge": [_P, _P, _I32, _P],
    "ts_nstep_return": [_P, _P, _P, _P, _I64, _I64, _I32, _D, _P, C.c_int, _P],
    "ts_buffer_end_flags": [_P, _P, _P, _P, _I64, _P, _P],
    "ts_value_mask_rows": [_P, _P, _P, _I64, _I64, _P],
    "ts_next_index": [_P, _I64, _P, _I64, _P, _P, _P, _P, _P],
    "ts_prev_index": [_P, _I64, _P, _I64, _P, _P, _P, _P, _P],
    "ts_stack_next_indices": [_P, _I64, _I32, _P, _I64, _P, _P, _P, _P, _P],
    "ts_unfinished_index": [_P, _I64, _P, _P, _P, _P, _P, _P, _P],
    "ts_sample_all_indices": [_P, _I64, _P, _P, _P, _P, _P, _I64, _P, _P],
    "ts_mark_members": [_P, _I64, _P, _P, _I64, _P, _I64, _P, _P],
    "ts_gather_rows": [_P, _I64, _P, _I64, _P, _P],
    "ts_scatter_rows": [_P, _I64, _P, _I64, _P, _P],
    "ts_segtree_setitem": [_P, _I64, _P, _P, C.c_int, _I64, _P],
    "ts_segtree_reduce": [_P, _I64, _I64, _I64, _P, _P],
    "ts_segtree_prefix_sum_idx": [_P, _I64, _P, _I64, _P, _P],
    "ts_segtree_sample": [_P, _I64, _P, _I64, _P, _P],
    "ts_prio_update_weight": [_P, _I64, _P, _P, C.c_int, _I64, _D, _D, _P, _P],
    "ts_prio_get_weight": [_P, _I64, _P, _I64, _P, _D, C.c_int, _P, _P],
    "ts_critic_forward": [_P, C.POINTER(ActorCriticDesc), _P, _P, _P, _P, _I64, _P],
    "ts_actor_logp": [_P, C.POINTER(ActorCriticDesc), _P, _P, _I64, _P, _P, _P],
    "ts_ppo_grad": [_P, C.POINTER(ActorCriticDesc), C.POINTER(PPOHParams), _P, _P, _P, _P, _P, _P, _P,
                    _I64, _I64, _I64, _P, _P, C.POINTER(_I32), _P],
    "ts_grad_reduce": [_P, _I32, C.POINTER(ActorCriticDesc), _P, _P],
    "ts_minibatch_adv_sums": [_P, _P, _I64, _I64, _P, _P],
    "ts_adv_moments_finalize": [_P, _I64, _P, _P],
    "ts_clip_adam_step": [_P, _P, _P, _I32, _P, _P, _P, C.POINTER(ActorCriticDesc), C.POINTER(PPOHParams), _P, _P],
    "ts_ppo_update": [_P, _P, _P, _P, _P, _P, C.POINTER(ActorCriticDesc), C.POINTER(PPOHParams),
                      _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _P, _I32,
                      C.POINTER(_I64), _I32, _I32, _D, _D, _P, _D, _P, _P, _P, _P, _P, _P],
    "ts_peer_alloc": [_I64, C.POINTER(C.c_void_p), _P],
    "ts_peer_open": [_P, C.POINTER(C.c_void_p)],
    "ts_peer_close": [_P],
    "ts_peer_free": [_P],
    "ts_epoch_adv_sums": [_P, _P, _I64, _I64, _I64, _I32, _P, _P],
    "ts_epoch_adv_finalize": [_P, _I64, _I64, _I64, _I32, _I32, _P, _P],
    "ts_ppo_epoch_multi": [_P, _P, _P, _P, _P, _P, C.POINTER(ActorCriticDesc), C.POINTER(PPOHParams),
                           _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I32, _P, _P, _P, _I32, _I32,
                           C.POINTER(C.c_void_p), _P],
    "ts_host_mt19937_permutation": [_P, C.POINTER(_I32), _I64, _P],
    "ts_host_perm_job_start": [_P, _I32, _I64, _I32, _P, _I32, C.POINTER(C.c_void_p)],
    "ts_host_perm_job_wait": [_P, _I32],
    "ts_host_perm_job_finish": [_P, _P, C.POINTER(_I32)],
    "ts_host_perm_feed_start": [_P, _P, _P, _I64, _I32, C.POINTER(C.c_void_p)],
    "ts_host_perm_feed_wait_row": [_P, _I32, _P],
    "ts_host_perm_feed_finish": [_P],
    "ts_make_permutation": [C.c_uint64, _I32, _I32, _I64, _P, _P],
    "ts_narrow_i64_i32": [_P, _I64, _P, _P],
    # layered networks of the off-policy algorithms (net_gemm.cu / net_ops.cu)
    "ts_net_gemm": [_P, _I64, _I32, _P, _I64, _I32, _P, _I64, _I32, _I32, _I32, _P, _I32, _P, _I64, _I32, _I32, _P, _I64, _P],
    "ts_ppo_rows": [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _P, _I64, _P, _P, _P, _P, _P, _P, _P],
    "ts_ppo_rows_stats": [_P, _I64, _P, _P, _P],
    "ts_net_colsum": [_P, _I64, _I32, _I32, _P, _I32, _P],
    "ts_stack_prev_indices": [_P, _I64, _I32, _P, _I64, _P, _P, _P, _P, _P],
    "ts_im2col_u8": [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _D, _P, _P],
    "ts_im2col_f32": [_P, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P],
    "ts_col2im_f32": [_P, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P, _P],
    "ts_nhwc_to_nchw_flat": [_P, _I32, _I32, _I32, _P, _P],
    "ts_nchw_flat_to_nhwc": [_P, _I32, _I32, _I32, _P, _P, _P],
    "ts_concat2": [_P, _I32, _P, _I32, _I64, _P, _P],
    "ts_squashed_gaussian": [_P, _I64, _P, _I64, _I32, C.c_float, C.c_float, C.c_float, _P, _P, _P, _P],
    "ts_squashed_gaussian_bwd": [_P, _I64, _P, _P, _P, _P, _I64, _I32, C.c_float, C.c_float, C.c_float, C.c_float, _P, _P],
    "ts_critic_mse": [_P, _P, _P, _I64, _P, _P, _P, _P],
    "ts_dqn_loss": [_P, _P, _P, _P, _I64, _I32, C.c_float, _P, _P, _P, _P],
    "ts_dqn_target": [_P, _P, _I64, _I32, _I32, _P, _P],
    "ts_sac_target": [_P, _P, _P, C.c_float, _I64, _P, _P],
    "ts_sac_actor_q_grad": [_P, _P, _P, C.c_float, _I64, _P, _P, _P, _P],
    "ts_det_actor_head": [_P, _I64, _I64, _I32, C.c_float, _P, C.c_float, C.c_float, _P, _P],
    "ts_det_actor_head_bwd": [_P, _I64, _P, _I64, _I32, C.c_float, _P, _P],
    "ts_det_actor_q_grad": [_P, _I64, _P, _P, _P],
    "ts_mean": [_P, _I64, _P, _P],
    "ts_adam_step": [_P, _P, _P, _P, _I64, _I64, _D, _D, _D, _D, _D, _D, _P, _P],
    "ts_adam_step_dev": [_P, _P, _P, _P, _I64, _P, _D, _D, _D, _D, _D, _D, _P, _P],
    "ts_polyak_update": [_P, _P, _I64, _D, _P],
}
# diagnostics build only (libts_b200_diag.so, tools/): not part of the product library
DIAG_SIGNATURES: dict[str, list[Any]] = {
    "ts_tc_timeline": [_I32, _P],
    "ts_umma_selftest": [_P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P],
}
DIAG_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libts_b200_diag.so")


def use_diagnostics_library() -> C.CDLL:
    """Make the process-wide library the DIAGNOSTICS build (phase timeline, tcgen05 self-test); tools/ only."""
    global _lib
    if not os.path.exists(DIAG_LIB_PATH):
        raise ExtensionMissingError(f"{DIAG_LIB_PATH} not found: build it with `python -m tianshou_b200.csrc.build --diag`")
    _lib = None
    lib = load_library(DIAG_LIB_PATH)
    for name, argtypes in DIAG_SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    _lib = lib
    return lib

OTHER_SYMBOLS = ["ts_version", "ts_last_error", "ts_launch_count", "ts_reset_launch_count",
                 "ts_gae_workspace_bytes", "ts_ppo_partial_rows", "ts_ppo_weight_image_bytes",
                 "ts_ppo_peer_buffer_bytes", "ts_net_gemm_workspace_floats"]

_lib: C.CDLL | None = None


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen the C-ABI library and attach prototypes.  Raises ExtensionMissingError loudly."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ExtensionMissingError(
            f"{p} not found: build it with `python -m tianshou_b200.csrc.build` "
            "(nvcc, sm_100a).  tianshou_b200 has no CPU fallback."
        )
    lib = C.CDLL(p)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.ts_version.restype = C.c_int
    lib.ts_last_error.restype = C.c_char_p
    lib.ts_launch_count.restype = C.c_int64
    lib.ts_reset_launch_count.restype = None
    lib.ts_gae_workspace_bytes.argtypes = [_I64]
    lib.ts_gae_workspace_bytes.restype = C.c_size_t
    lib.ts_ppo_partial_rows.restype = C.c_int32
    lib.ts_ppo_weight_image_bytes.argtypes = [C.POINTER(ActorCriticDesc)]
    lib.ts_ppo_weight_image_bytes.restype = C.c_int64
    lib.ts_ppo_peer_buffer_bytes.argtypes = [C.POINTER(ActorCriticDesc), _I32]
    lib.ts_ppo_peer_buffer_bytes.restype = C.c_int64
    lib.ts_net_gemm_workspace_floats.argtypes = [_I32, _I32, _I32]
    lib.ts_net_gemm_workspace_floats.restype = C.c_int64
    if path is None:
        _lib = lib
    return lib


def require_cuda() -> None:
    if not torch.cuda.is_available():
        raise ExtensionMissingError(
            "tianshou_b200 device path called without a CUDA device: there is no CPU fallback."
        )


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load_library().ts_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (status {status}): {msg}")


def ptr(t: torch.Tensor | None) -> int | None:
    """Raw device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda, "device pointer requested for a host tensor"
    assert t.is_contiguous(), "kernels take dense tensors"
    return t.data_ptr()


def stream_ptr(device: torch.device | None = None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def call(name: str, *args: Any) -> None:
    lib = load_library()
    check(getattr(lib, name)(*args), name)


def launch_count() -> int:
    return int(load_library().ts_launch_count())


def reset_launch_count() -> None:
    load_library().ts_reset_launch_count()


def to_device(a: np.ndarray | torch.Tensor, device: torch.device, dtype: torch.dtype | None = None,
              non_blocking: bool = False) -> torch.Tensor:
    """numpy / tensor -> contiguous device tensor (bool arrays become uint8 views)."""
    if isinstance(a, np.ndarray):
        if a.dtype == np.bool_:
            a = a.view(np.uint8)
        t = torch.from_numpy(np.ascontiguousarray(a))
    else:
        t = a
        if t.dtype == torch.bool:
            t = t.view(torch.uint8)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.to(device, non_blocking=non_blocking).contiguous()
