"""ctypes binding of ``libdgtd_ops.so`` (declared in ``include/dgtd_ops.h``).

There is deliberately no fallback: if the shared object is missing or a call fails, a
``RuntimeError`` is raised (the reference's extension raises the same way through
``AT_ERROR`` -> ``RuntimeError``, twig/ops/src/ms_deform_attn.h:35-38).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_void_p
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdgtd_ops.so")

F32, BF16 = 0, 1
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2

_P, _I, _L, _F = c_void_p, c_int, c_int64, c_float

# name -> argument types (return type is always int unless listed in _RESTYPES)
SIGNATURES = {
    "dgtd_version": [],
    "dgtd_last_error": [],
    "dgtd_launch_count": [],
    "dgtd_surface_normals_fwd": [_P, _P, _I, _I, _I, _P],
    "dgtd_lowpass_projector": [_P, _P, _I, _I, _P],
    "dgtd_fft_highpass_fwd": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "dgtd_fft_highpass_tc3_fwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "dgtd_diffusion_front_fwd": [_P] * 11 + [_I] * 6 + [_P],
    "dgtd_message_passing_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P],
    "dgtd_message_passing_tiled_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _I, _P],
    "dgtd_message_passing_tiled_simt_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _I, _P],
    "dgtd_message_passing_tc_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _I, _P],
    "dgtd_pack_regressor": [_P, _P, _P, _I, _P],
    "dgtd_message_passing_regress_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _I, _I, _P],
    "dgtd_message_passing_bwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P],
    "dgtd_conv1x1_nchw_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_conv1x1_nchw_bwd": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_resize_bilinear_nchw_bwd": [_P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_resize_nchw_fwd": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_resize_sigmoid_sized_fwd": [_P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_layer_norm_fwd": [_P, _P, _P, _P, _L, _I, _L, _F, _P],
    "dgtd_stem_fwd": [_P, _P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _P],
    "dgtd_ln_patchify_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "dgtd_dwconv7_ln_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "dgtd_dwconv7_ln_tma_fwd": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "dgtd_linear_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_dwconv7_stats_tma_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _P],
    "dgtd_linear_ln_fwd": [_P, _P, _P, _P, _P, _F, _P, _I, _I, _I, _P],
    "dgtd_linear_tf32_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_linear_lnfold_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_linear_residual_fwd": [_P, _P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_convnext_mlp_fused_fwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _P],
    "dgtd_fusion_sum_fwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "dgtd_conv_nhwc_fwd": [_P, _P, _P, _P] + [_I] * 15 + [_P],
    "dgtd_conv_nhwc_grouped_fwd": [_P, _P, _P, _P] + [_I] * 16 + [_L, _I, _L, _P],
    "dgtd_resize_nhwc_fwd": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_linear_dgrad": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_linear_wgrad": [_P, _P, _P, _P, _P] + [_I] * 13 + [_P],
    "dgtd_linear_wgrad_ws_floats": [_I, _I, _I],
    "dgtd_colsum": [_P, _P, _I, _P, _P, _I, _I, _P],
    "dgtd_layer_scale_finalize": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P],
    "dgtd_gelu_fwd": [_P, _P, _L, _P],
    "dgtd_relu_bwd": [_P, _P, _P, _L, _P],
    "dgtd_ln_rows_bwd": [_P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _P],
    "dgtd_ln_rows_bwd_ws_floats": [_L, _I],
    "dgtd_dwconv7_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_dwconv7_wgrad": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_stem_patchify": [_P, _P, _I, _P, _I, _I, _I, _I, _P],
    "dgtd_stem_unpatchify": [_P, _P, _I, _I, _I, _P],
    "dgtd_patchify2": [_P, _P, _I, _I, _I, _I, _P],
    "dgtd_unpatchify2": [_P, _P, _I, _I, _I, _I, _P],
    "dgtd_resize_nhwc_bwd": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_transpose_op": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_colsum_bf16": [_P, _P, _P, _I, _I, _P],
    "dgtd_eltwise_colsum_ws_floats": [_I, _I],
    "dgtd_eltwise_colsum": [_P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _P],
    "dgtd_wgrad_tc_ws_floats": [_I, _I, _I],
    "dgtd_wgrad_tc_mn": [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_ln_rows_fwd": [_P, _P, _P, _P, _I, _L, _I, _F, _P],
    "dgtd_ln_tokens_fwd": [_P, _P, _I, _P, _P, _P, _P, _I, _L, _I, _F, _P],
    "dgtd_patchify_tokens_fwd": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_dwconv3_gelu_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_dwconv3_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_attention_fwd": [_P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "dgtd_attention_bwd_ws_floats": [_I, _I, _I, _I],
    "dgtd_attention_bwd": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "dgtd_dwconv3_gelu_bwd_ws_floats": [],
    "dgtd_dwconv3_gelu_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_boundary_weight_fwd": [_P, _P, _I, _I, _I, _P],
    "dgtd_structure_loss_ws_floats": [_I, _L],
    "dgtd_structure_loss_fwd": [_P, _P, _P, _P, _P, _P, _I, _L, _P],
    "dgtd_structure_loss_bwd": [_P, _P, _P, _P, _P, _P, _I, _L, _P],
    "dgtd_col2im_nhwc": [_P, _I, _I, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_im2col_nhwc": [_P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_group_sum": [_P, _I, _P, _L, _I, _I, _I, _P],
    "dgtd_cast_fwd": [_P, _P, _L, _I, _I, _P],
    "dgtd_nhwc_to_nchw_fwd": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_nchw_to_nhwc_fwd": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_conv_nhwc_affine_fwd": [_P, _P, _P, _P, _P, _P, _I, _P] + [_I] * 12 + [_P],
    "dgtd_channel_sums_chunks": [_I],
    "dgtd_channel_sums_fwd": [_P, _I, _P, _I, _I, _I, _P],
    "dgtd_channel_gate_fwd": [_P, _I, _I, _P, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_gated_sum_fwd": [_P, _I, _P, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_resize_nhwc_ld_fwd": [_P, _I, _P, _I] + [_I] * 7 + [_P],
    "dgtd_copy_channels_fwd": [_P, _I, _P, _I, _L, _I, _P],
    "dgtd_head1_fwd": [_P, _I, _P, _P, _P, _L, _I, _I, _P],
    "dgtd_sigmoid_fwd": [_P, _P, _L, _P],
    "dgtd_cast_pad_act_fwd": [_P, _I, _P, _P, _L, _I, _I, _P],
    "dgtd_conv3x3_tc_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "dgtd_im2col_act_fwd": [_P, _I, _P, _P] + [_I] * 9 + [_P],
    "dgtd_col_stats_ws_bytes": [_L, _I],
    "dgtd_bn_train_fwd": [_P, _I, _P, _P, _P, _P, _F, _F, _P, _I, _P, _P, _P, _L, _I, _P],
    "dgtd_bn_apply_fwd": [_P, _I, _P, _P, _P, _P, _P, _I, _L, _I, _P],
    "dgtd_bn_train_bwd": [_P, _I, _P, _I, _P, _P, _P, _P, _I, _P, _P, _P, _I, _L, _I, _P],
    "dgtd_prelu_fwd": [_P, _P, _P, _L, _P],
    "dgtd_prelu_bwd_ws_bytes": [_L],
    "dgtd_prelu_bwd": [_P, _P, _P, _P, _P, _P, _L, _P],
    "dgtd_channel_dot_fwd": [_P, _I, _P, _I, _P, _I, _I, _I, _P],
    "dgtd_gate_bwd_ws_floats": [_I, _I, _I, _I],
    "dgtd_gate_bwd": [_P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dgtd_gated_bwd": [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "dgtd_head1_bwd": [_P, _P, _I, _P, _P, _I, _P, _P, _P, _L, _I, _P],
    "dgtd_resize_nhwc_ld_bwd": [_P, _I, _P, _I] + [_I] * 7 + [_P],
    "dgtd_ssim_loss_ws_floats": [_L],
    "dgtd_ssim_loss_fwd": [_P, _P, _P, _P, _I, _I, _I, _P],
    "dgtd_adamw_slice_bytes": [],
    "dgtd_adamw_step": [_P, _P, _P, _P, _P, _I, _F, _F, _F, _I, _F, _F, _P],
    "dgtd_sod_metrics_ws_bytes": [_I, _I, _I],
    "dgtd_sod_metrics_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _P],
    "dgtd_sod_wfm_ws_bytes": [_I, _I, _I],
    "dgtd_sod_wfm_fwd": [_P, _P, _P, _P, _I, _I, _I, _P],
    "dgtd_sod_metrics_sized_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "dgtd_sod_wfm_sized_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _P],
}
_RESTYPES = {"dgtd_last_error": c_char_p, "dgtd_launch_count": c_int64, "dgtd_sod_metrics_ws_bytes": c_int64,
             "dgtd_sod_wfm_ws_bytes": c_int64,
             "dgtd_col_stats_ws_bytes": c_int64, "dgtd_attention_bwd_ws_floats": c_int64, "dgtd_dwconv3_gelu_bwd_ws_floats": c_int64, "dgtd_gate_bwd_ws_floats": c_int64, "dgtd_prelu_bwd_ws_bytes": c_int64}

_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """Load (once) and type the library.  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m dgtd_b200.twig.ops.build` "
            "(there is no CPU or PyTorch fallback for the texture-diffusion kernels)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so lost a symbol
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, c_int)
    if lib.dgtd_version() != 100:
        raise RuntimeError(f"libdgtd_ops.so version {lib.dgtd_version()} != 100 (stale build?)")
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().dgtd_last_error()
    return msg.decode() if msg else ""


def launch_count() -> int:
    return int(load().dgtd_launch_count())


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise TypeError(f"dgtd ops support float32 / bfloat16 only, got {dt}")


_PROF = {"on": False, "events": []}


def enable_profile(on: bool = True) -> None:
    """Per-entry-point CUDA-event timing (tools/op_profile.py); off by default."""
    _PROF["on"] = bool(on)
    _PROF["events"] = []


def profile_summary() -> dict:
    torch.cuda.synchronize()
    out = {}
    for name, a, b in _PROF["events"]:
        e = out.setdefault(name, [0, 0.0])
        e[0] += 1
        e[1] += a.elapsed_time(b)
    return out


def call(name: str, *args) -> None:
    """Invoke an entry point; raise RuntimeError(dgtd_last_error()) on a non-zero return."""
    lib = load()
    if _PROF["on"]:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = getattr(lib, name)(*args)
        b.record()
        _PROF["events"].append((name, a, b))
    else:
        rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {last_error()}")


def check_cuda(*tensors: Optional[torch.Tensor]) -> None:
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("dgtd ops run on CUDA tensors only (no CPU fallback); got a "
                               f"{t.device} tensor")
        if not t.is_contiguous():
            raise RuntimeError("dgtd ops need contiguous tensors")
