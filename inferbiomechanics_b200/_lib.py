"""ctypes binding of libibm_b200.so (the C ABI declared in include/ibm_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is missing the import
of any compute entry point raises, telling the user to build it.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int32, c_int64, c_size_t, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libibm_b200.so")

ACT = {"none": 0, None: 0, "relu": 1, "sigmoid": 2, "tanh": 3, "elu": 4, "silu": 5}
F32, BF16 = 0, 1
OPT_KIND = {"rmsprop": 0, "adam": 1, "sgd": 2, "adagrad": 3, "adadelta": 4, "adamax": 5}

P = c_void_p
_i32, _i64, _u64, _f = c_int32, c_int64, c_uint64, c_float

# name -> argtypes  (restype is int for all but the few listed in _SPECIAL)
SIGNATURES = {
    "ibm_window_valid_mask": [P, P, P, P, _i64, _i32, _i32, P, P],
    "ibm_pack_windows": [P, _i64, _i32, P, _i64, _i32, _i32, P, P, _i64, _i64, _i64, P],
    "ibm_pack_inputs": [P, P, _i32, _i64, _i32, P, P, _i64, _i64, _i64, P],
    "ibm_pack_channel_major": [P, P, _i32, _i64, _i32, P, _i32, P, _i64, P],
    "ibm_pack_labels": [P, _i64, _i32, P, P, P, _i64, _i32, _i32, _i32, P, _i64, P],
    "ibm_regression_loss_fwd": [P, P, P, P, _i64, _i64, P, _f, P, P, P],
    "ibm_regression_loss_bwd": [P, P, P, P, _i64, _i64, P, _f, P, P, P, _i32, P],
    "ibm_sqdiff_mean_vector": [P, _i64, _i64, P, _i64, _i64, _i64, _i64, _i32, P, P, P],
    "ibm_sqdiff_mean_vector_bwd": [P, _i64, _i64, P, _i64, _i64, _i64, _i64, _i32, P, P, P, P],
    "ibm_mask_by_threes": [P, _i64, _i64, _i64, _i64, _i32, _f, P, P],
    "ibm_mean_norm_error": [P, _i64, _i64, P, _i64, _i64, _i64, _i64, _i32, _i32, _i32, P, P, P],
    "ibm_q_sample": [P, P, P, P, P, _i64, _i64, P, P, _i64, _u64, _u64, P, P],
    "ibm_ddpm_posterior_step": [P, _i64, P, P, P, P, P, P, _i64, P, P, _i64, _u64, _u64, P, P],
    "ibm_ddpm_respaced_step": [P, _i64, P, P, P, P, P, P, _i64, P, P, _i64, _u64, _u64, P, P, P],
    "ibm_ddpm_guided_step": [P, _i64, P, P, P, P, P, P, _i64, P, P, _i64, _u64, _u64, P, P, _f, P],
    "ibm_ddpm_inpaint_step": [P, _i64, P, P, P, P, P, P, _i64, P, P, _i64, _u64, _u64, P, P, _f, _i32, P, P, P],
    "ibm_ddpm_multistep_step": [P, _i64, P, P, P, P, P, P, _i64, P, P, P, _i64, P, _f, _i32, P, P, P],
    "ibm_cond_dropout": [P, _i64, _i64, _i32, _i32, _i32, _f, _u64, _u64, P, P],
    "ibm_ensemble_score": [P, _i32, _i64, _i32, P, _i32, _f, P, P, P, P, P],
    "ibm_timestep_embed": [P, _i32, _i64, _i32, P, P],
    "ibm_add_time_pos": [P, _i64, P, _i64, P, _i64, _i32, _i32, P, P],
    "ibm_add_time_pos_bwd": [P, _i64, P, _i64, P, _i64, _i32, _i32, P, P],
    "ibm_gemm_bf16": [P, _i64, _i32, P, _i64, _i32, _i64, _i64, _i64, P, _i32, P, _i64, _i32, P, _i64, _i32, _i32,
                      _i32, _i32, P, P, _i64, _i32, P],
    "ibm_colsum_bf16": [P, _i64, _i64, _i64, P, P],
    "ibm_act_fwd": [P, P, _i64, _i32, P],
    "ibm_act_bwd": [P, P, P, _i64, _i32, P],
    "ibm_cast_f32_bf16": [P, P, _i64, P],
    "ibm_cast_bf16_f32": [P, P, _i64, P],
    "ibm_cast_pad_f32_bf16": [P, _i64, P, _i64, _i64, _i64, P],
    "ibm_conv_weight_to_gemm": [P, _i32, _i32, _i32, _i32, P, P],
    "ibm_conv_wgrad_from_gemm": [P, _i32, _i32, _i32, _i32, P, _i32, P],
    "ibm_replicate_pad_rows": [P, _i64, _i64, _i32, _i32, _i32, P],
    "ibm_fold_pad_rows": [P, _i64, _i64, _i32, _i32, _i32, P],
    "ibm_dropout_bf16": [P, P, _i64, _f, _u64, _u64, P],
    "ibm_dropout_bf16_dev": [P, P, _i64, _f, _u64, _u64, P, _i64, P],
    "ibm_conv_weight_to_dgrad": [P, _i32, _i32, _i32, _i32, P, P],
    "ibm_batchnorm_fwd": [P, _i64, P, _i64, _i64, _i32, P, P, P, P, P, P, _i32, _f, _f, P, P],
    "ibm_batchnorm_bwd": [P, _i64, P, _i64, P, _i64, _i64, _i32, P, P, P, _i32, _f, P, _i64, _i32, P, P, P, P, P],
    "ibm_layernorm_fwd": [P, P, _i64, P, P, _i64, _i32, _f, P, P, P],
    "ibm_layernorm_bwd": [P, P, _i64, P, P, P, _i64, _i32, P, P, P, P, P],
    "ibm_attention_fwd": [P, _i64, P, _i64, P, _i64, P, _i64, _i64, _i32, _i32, _i32, _i32, _f, P],
    "ibm_attention_bwd": [P, _i64, _i64, P, _i64, P, _i64, _i32, _i32, _i32, _f, P, P],
    "ibm_expand_rows_bf16": [P, _i64, _i32, _i64, _i32, P, _i32, P, _i64, P, _i32, P],
    "ibm_attention_bwd_long": [P, _i64, P, _i64, P, _i64, P, _i64, P, _i64, P, _i64, P, _i64, P, _i64, _i64, _i32, _i32, _i32, _i32, _f,
                               P, P, P, P],
    "ibm_optimizer_step_dev": [_i32, P, P, P, P, P, _i64, _f, _f, P, P],
    "ibm_optimizer_step_ema": [_i32, P, P, P, P, P, P, _i64, _f, _f, _f, _i64, P, P],
    "ibm_grad_clip_coef": [P, _i64, _f, _f, P, P, P, P, P],
    "ibm_optimizer_step_sched": [_i32, P, P, P, P, P, P, _i64, _f, _f, _f, _i64, P, P, _i32, _i64, _i64, _f, P],
    "ibm_counter_add": [P, _i64, P],
    "ibm_optimizer_step": [_i32, P, P, P, P, P, _i64, _f, _f, _i64, P],
    "ibm_device_check": [_i32],
    "ibm_debug_gemm_max_clusters": [_i32],
    "ibm_set_walk_order": [_i32],
}
_SPECIAL = {
    "ibm_version": ([], c_int32),
    "ibm_last_error": ([c_char_p, c_size_t], c_size_t),
    "ibm_workspace_bytes": ([], c_size_t),
    "ibm_batchnorm_workspace_floats": ([c_int32], c_size_t),
}
ALL_SYMBOLS = sorted(list(SIGNATURES) + list(_SPECIAL))

_lib = None


class IbmError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IbmError(
            f"{LIB_PATH} not found. inferbiomechanics_b200 has no CPU or PyTorch fallback: build the sm_100a "
            f"extension first with `python -m inferbiomechanics_b200.build` (or __graft_entry__.build()).")
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = c_int32
    for name, (argtypes, restype) in _SPECIAL.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def last_error() -> str:
    buf = ctypes.create_string_buffer(1024)
    load().ibm_last_error(buf, 1024)
    return buf.value.decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = last_error()
        if rc == 1:
            raise ValueError(f"{what}: {msg}")
        raise IbmError(f"{what} failed (code {rc}): {msg}")


# launch counter: bench.py reports how many of OUR kernels ran inside the timed region
launch_count = 0


def call(name: str, *args) -> None:
    global launch_count
    launch_count += 1
    check(getattr(load(), name)(*args), name)
