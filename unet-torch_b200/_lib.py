"""ctypes binding of libb200unet.so (the C ABI declared in include/b200unet.h).

The product path has NO fallback: if the shared library is missing or fails to load, importing the kernels
raises. `build.py` produces the library in-tree (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_double, c_float, c_int, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200unet.so")

_P = c_void_p
_I = c_int
_L = c_int64
_F = c_float
_D = c_double

# name -> (restype, argtypes); mirrors include/b200unet.h one to one
SIGNATURES = {
    "b200unet_version": (c_int, []),
    "b200unet_last_error": (ctypes.c_char_p, []),
    "b200unet_launch_count": (c_int64, []),
    "b200unet_tile_h": (c_int, []),
    "b200unet_tile_w": (c_int, []),
    "b200unet_prep_conv3x3_weight": (c_int, [_P, _P, _P, _I, _I, _P]),
    "b200unet_prep_convt2x2_weight": (c_int, [_P, _P, _P, _I, _I, _P]),
    "b200unet_set_kernel_choice": (c_int, [_I, _I, _I]),
    "b200unet_conv3x3_stat_rows": (c_int, [_I, _I, _I, _I, _I]),
    "b200unet_conv3x3_igemm": (c_int, [_P, _I, _P, _P, _I, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv3x3_dgrad_bnred_rows": (c_int, [_I, _I, _I, _I, _I]),
    "b200unet_conv3x3_igemm_bnred": (c_int, [_P, _I, _P, _P, _I, _P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv3x3_bn_relu_igemm": (c_int, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv1x1_c64_bn_relu_igemm": (c_int, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_convt2x2_fprop": (c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_convt2x2_dgrad": (c_int, [_P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv3x3_wgrad_workspace_floats": (c_int64, [_I, _I, _I, _I, _I]),
    "b200unet_conv3x3_wgrad": (c_int, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_convt2x2_wgrad_workspace_floats": (c_int64, [_I, _I, _I, _I, _I]),
    "b200unet_convt2x2_wgrad": (c_int, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_first_im2col": (c_int, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_prep_first_weight": (c_int, [_P, _P, _I, _I, _P]),
    "b200unet_conv3x3_first_igemm": (c_int, [_P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv3x3_first_bn_relu_igemm": (c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv3x3_first_tc_wgrad_workspace_floats": (c_int64, [_I, _I, _I, _I]),
    "b200unet_conv3x3_first_tc_wgrad": (c_int, [_P, _P, _I, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv1x1_c64_stat_rows": (c_int, [_I, _I, _I, _I]),
    "b200unet_conv1x1_c64_igemm": (c_int, [_P, _I, _P, _P, _I, _P, _I, _I, _I, _I, _P]),
    "b200unet_conv1x1_c64_wgrad_workspace_floats": (c_int64, [_I, _I, _I, _I]),
    "b200unet_conv1x1_c64_wgrad": (c_int, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv3x3_first_fprop": (c_int, [_P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv3x3_first_wgrad_workspace_floats": (c_int64, [_I, _I, _I, _I, _I]),
    "b200unet_conv3x3_first_wgrad": (c_int, [_P, _P, _I, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_head_fprop": (c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_head_bwd_workspace_floats": (c_int64, [_I, _I, _I, _I, _I]),
    "b200unet_head_bwd": (c_int, [_P, _P, _I, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_head_many_fprop": (c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_head_many_bwd_workspace_floats": (c_int64, [_I, _I, _I, _I, _I]),
    "b200unet_head_many_bwd": (c_int, [_P, _P, _I, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_bn_reduce_partials": (c_int, [_P, _L, _I, _P, _P]),
    "b200unet_fold_rows": (c_int, [_P, _L, _I, _P, _I, _P]),
    "b200unet_bn_finalize": (c_int, [_P, _D, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P, _I, _P]),
    "b200unet_bn_reduce_finalize": (c_int, [_P, _L, _I, _D, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P, _P, _P]),
    "b200unet_bn_eval_affine": (c_int, [_P, _P, _P, _P, _F, _P, _P, _I, _P]),
    "b200unet_bn_eval_stats": (c_int, [_P, _P, _F, _P, _P, _I, _P]),
    "b200unet_bn_relu_fwd": (c_int, [_P, _I, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_bn_bwd_workspace_floats": (c_int64, [_I, _I, _I, _I]),
    "b200unet_bn_relu_bwd_reduce_rows": (c_int, [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_bn_relu_bwd_reduce": (c_int, [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_bn_relu_bwd_apply": (
        c_int,
        [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _D, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P],
    ),
    "b200unet_partial_colsum": (c_int, [_P, _L, _I, _I, _I, _P, _P]),
    "b200unet_bn_relu_fwd_floor": (c_int, [_P, _I, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_bn_relu_bwd_reduce_rows_floor": (c_int, [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_bn_relu_bwd_reduce_floor": (c_int, [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_bn_relu_bwd_apply_floor": (
        c_int, [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _D, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_pad_strip_zero": (c_int, [_P, _I, _I, _I, _I, _I, _P]),
    "b200unet_pad_strip_sub_colsum": (c_int, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "b200unet_maxpool2x2_fwd_floor": (c_int, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P]),
    "b200unet_maxpool2x2_fwd": (c_int, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P]),
    "b200unet_nhwc_copy": (c_int, [_P, _I, _P, _I, _L, _I, _P]),
    "b200unet_nhwc_add": (c_int, [_P, _I, _P, _I, _P, _I, _L, _I, _P]),
    "b200unet_channel_sum_workspace_floats": (c_int64, [_I]),
    "b200unet_channel_sum": (c_int, [_P, _I, _P, _P, _L, _I, _P]),
    "b200unet_dropout_partial_rows": (c_int, [_I, _I, _I, _I]),
    "b200unet_dropout_mul": (c_int, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _L, _F, _P, _I, _I, _P]),
    "b200unet_loss_sums_doubles": (c_int, []),
    "b200unet_loss_sums_doubles_n": (c_int64, [_I]),
    "b200unet_loss_sums_saved_doubles_n": (c_int64, [_I]),
    "b200unet_loss_ce_dice_fwd": (c_int, [_P, _P, _P, _P, _P, _I, _I, _L, _I, _P]),
    "b200unet_loss_ce_dice_bwd": (c_int, [_P, _P, _P, _P, _P, _I, _I, _L, _I, _P]),
    "b200unet_mse_fwd": (c_int, [_P, _P, _P, _P, _L, _I, _P]),
    "b200unet_mse_bwd": (c_int, [_P, _P, _P, _P, _L, _I, _P]),
    "b200unet_softmax_argmax": (c_int, [_P, _P, _I, _I, _L, _P]),
    "b200unet_gen_conv3x3": (c_int, [_P, _L, _P, _P, _L, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_gen_conv3x3_wgrad": (c_int, [_P, _L, _P, _L, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_gen_channel_stats": (c_int, [_P, _L, _P, _I, _I, _I, _P]),
    "b200unet_gen_bn_relu_fwd": (c_int, [_P, _L, _P, _P, _P, _L, _I, _I, _I, _P]),
    "b200unet_gen_maxpool2x2": (c_int, [_P, _L, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_gen_unpool_add": (c_int, [_P, _P, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_gen_bn_relu_bwd_reduce": (c_int, [_P, _L, _P, _L, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "b200unet_gen_bn_relu_bwd_apply": (c_int, [_P, _L, _P, _L, _P, _P, _P, _P, _P, _P, _D, _P, _P, _L, _P, _P, _I, _I, _I, _P]),
    "b200unet_gen_convt2x2_fprop": (c_int, [_P, _L, _P, _P, _P, _L, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_gen_convt2x2_dgrad": (c_int, [_P, _L, _P, _P, _L, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_gen_convt2x2_wgrad": (c_int, [_P, _L, _P, _L, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_gen_conv1x1_fwd": (c_int, [_P, _L, _P, _P, _P, _I, _I, _I, _L, _P]),
    "b200unet_gen_conv1x1_bwd": (c_int, [_P, _P, _L, _P, _P, _L, _P, _P, _I, _I, _I, _L, _P]),
    "b200unet_gen_mul": (c_int, [_P, _L, _P, _I, _L, _P]),
    "b200unet_gen_bn_act_fwd": (c_int, [_P, _L, _P, _P, _P, _L, _I, _I, _I, _I, _P]),
    "b200unet_gen_bn_bwd_reduce": (c_int, [_P, _L, _P, _L, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_gen_bn_bwd_apply": (c_int, [_P, _L, _P, _L, _P, _P, _P, _P, _P, _P, _D, _P, _P, _L, _P, _P, _I, _I, _I, _I, _P]),
    "b200unet_gen_add_relu": (c_int, [_P, _P, _P, _L, _P]),
    "b200unet_gen_relu_bwd": (c_int, [_P, _P, _P, _L, _P]),
    "b200unet_gen_gate_fwd": (c_int, [_P, _L, _P, _P, _L, _I, _I, _L, _P]),
    "b200unet_gen_gate_bwd": (c_int, [_P, _L, _P, _L, _P, _P, _L, _P, _I, _I, _L, _P]),
    "b200unet_gen_add_inplace": (c_int, [_P, _L, _P, _L, _I, _L, _P]),
    "b200unet_znorm_workspace_bytes": (c_int64, [_I, _I]),
    "b200unet_znorm_to_chw": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_head_mask": (c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_head_sigmoid_mask": (c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
    "b200unet_head_density": (c_int, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
    "b200unet_head_many_mask": (c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "b200unet_head_many_density": (c_int, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
    "b200unet_nvl_buffer_bytes": (c_int64, []),
    "b200unet_nvl_allreduce_f64": (c_int, [_P, _P, _I, _P, _I, _I, _L, _P]),
    "b200unet_nvl_bn_sync_finalize": (c_int, [_P, _P, _P, _I, _I, _L, _D, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P, _I, _P]),
    "b200unet_nvl_rows_allreduce": (c_int, [_P, _L, _I, _P, _I, _I, _P, _P, _P]),
    "b200unet_nvl_bn_rows_sync_finalize": (c_int, [_P, _L, _I, _P, _I, _I, _D, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P, _P, _P]),
    "b200unet_nvl_set_timeout_ms": (c_int, [_L]),
    "b200unet_nvl_status": (c_int, [_P, _P, _P]),
    "b200unet_sgd_conv3x3_weight": (c_int, [_P, _P, _P, _P, _P, _I, _I, _F, _F, _F, _F, _I, _I, _P]),
    "b200unet_sgd_convt2x2_weight": (c_int, [_P, _P, _P, _P, _P, _I, _I, _F, _F, _F, _F, _I, _I, _P]),
    "b200unet_conv1x1_stat_rows": (c_int, [_I, _I, _I]),
    "b200unet_conv1x1_fprop": (c_int, [_P, _I, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_conv1x1_wgrad_workspace_floats": (c_int64, [_I, _I, _I, _I, _I]),
    "b200unet_conv1x1_wgrad": (c_int, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_convt2x2_stat_rows": (c_int, [_I, _I, _I]),
    "b200unet_convt2x2_fprop_stats": (c_int, [_P, _I, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "b200unet_gate_workspace_floats": (c_int64, [_I]),
    "b200unet_gate_stat_rows": (c_int, [_L, _I]),
    "b200unet_gate_psi_fwd": (c_int, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "b200unet_gate_apply_fwd": (c_int, [_P, _I, _P, _P, _P, _P, _I, _L, _I, _P]),
    "b200unet_gate_apply_bwd": (c_int, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _L, _I, _P]),
    "b200unet_gate_dx": (c_int, [_P, _I, _P, _P, _P, _P, _I, _L, _I, _P]),
    "b200unet_gate_bwd_reduce": (c_int, [_P, _I, _P, _I] + [_P] * 15 + [_D, _P, _P, _P, _L, _I, _P]),
    "b200unet_gate_bwd_apply": (c_int, [_P, _I, _P, _I] + [_P] * 15 + [_D] + [_P] * 10 + [_L, _I, _P]),
    "b200unet_sgemm_strided": (c_int, [_P, _P, _P, _P, _I, _I, _I, _L, _L, _L, _L, _L, _L, _I, _L, _L, _L, _I, _P]),
    "b200unet_sum_batches": (c_int, [_P, _P, _L, _I, _P]),
    "b200unet_sgd_small": (c_int, [_P, _P, _P, _P, _I, _F, _F, _F, _F, _I, _I, _P]),
    "b200unet_sgd_weights": (c_int, [_I, _P, _P, _P, _P, _P, _P, _P, _I, _F, _F, _F, _F, _I, _I, _P]),
    "b200unet_adam_weights": (c_int, [_I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _D, _D, _F, _F, _F, _F, _I, _P]),
    "b200unet_adam_conv3x3_weight": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _D, _D, _F, _F, _F, _F, _I, _P]),
    "b200unet_adam_convt2x2_weight": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _D, _D, _F, _F, _F, _F, _I, _P]),
    "b200unet_adam_small": (c_int, [_P, _P, _P, _P, _P, _I, _D, _D, _F, _F, _F, _F, _I, _P]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (once). Raises if it has not been built: there is no CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). The B200 U-Net path has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().b200unet_last_error().decode("utf-8", "replace")


def call(name: str, *args):
    """Call an int-returning entry point; non-zero -> RuntimeError carrying the library's message."""
    rc = getattr(load(), name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed (code {rc}): {last_error()}")


def query(name: str, *args):
    return getattr(load(), name)(*args)
