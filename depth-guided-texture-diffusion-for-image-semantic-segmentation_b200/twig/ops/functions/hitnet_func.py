"""Operator functions of the Hitnet iterative decoder (SURVEY.md 8f-2): Python side of csrc/hitnet_ops.cu,
same conventions as texture_diffusion_func.py (torch allocates, the library computes; NHWC fp32; a tensor
argument may be a channel slice `t[..., a:b]` of a wider tensor, which is how the reference's torch.cat
operands are produced in place)."""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from .. import capi
from ..capi import call, check_cuda, ptr, stream
from ...padded import PaddedBatch

__all__ = ["conv_affine", "conv_affine_tc", "conv3_tc", "channel_sums", "channel_gate", "gated_sum", "resize_ld", "copy_channels", "head1", "sigmoid",
           "resize_sigmoid_sized"]


def _on_cuda(*tensors: Optional[torch.Tensor]) -> None:
    """Like capi.check_cuda, but channel slices are allowed (their layout is checked by `_pitch`)."""
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(f"dgtd ops run on CUDA tensors only (no CPU fallback); got a {t.device} tensor")


def _pitch(t: torch.Tensor) -> int:
    """Pixel pitch of an NHWC tensor or channel slice (rows must be dense apart from the pitch)."""
    assert t.dtype == torch.float32 and t.stride(-1) == 1, "fp32 NHWC (slice) expected"
    ld = t.stride(-2)
    if t.dim() == 4:
        B, h, w, _ = t.shape
        assert t.stride(1) == w * ld and (B == 1 or t.stride(0) == h * w * ld), "not a channel slice of an NHWC tensor"
    return ld


def conv_affine(x: torch.Tensor, w: torch.Tensor, out_hw: Tuple[int, int], ks: int, stride: int, off: int,
                scale: Optional[torch.Tensor] = None, shift: Optional[torch.Tensor] = None,
                prelu: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """prelu(scale * conv(x) + shift) + residual; `w` packed (Cout, ks*ks*Cin) tap-major."""
    check_cuda(w, scale, shift, prelu)
    _on_cuda(x, residual, out)
    B, h, wd, Cin = x.shape
    Cout = w.shape[0]
    assert w.shape[1] == ks * ks * Cin, (tuple(w.shape), ks, Cin)
    oh, ow = out_hw
    if out is None:
        out = torch.empty(B, oh, ow, Cout, device=x.device, dtype=torch.float32)
    assert out.shape == (B, oh, ow, Cout)
    call("dgtd_conv_nhwc_affine_fwd", x.data_ptr(), ptr(w), ptr(scale), ptr(shift), ptr(prelu), ptr(residual),
         _pitch(residual) if residual is not None else 0, out.data_ptr(), B, h, wd, Cin, _pitch(x), oh, ow, Cout,
         _pitch(out), ks, stride, off, stream())
    return out




def _col_scratch(device: torch.device, numel: int) -> torch.Tensor:
    """bf16 im2col operand, reused by every conv of the decoder (stream-ordered producer / consumer pairs)."""
    from ...model.texture_diffuser import scratch_buffer      # capture-safe, per-stream (see its docstring)
    return scratch_buffer("hitnet_col", device, numel, torch.bfloat16)


def conv_affine_tc(x: torch.Tensor, w: torch.Tensor, out_hw: Tuple[int, int], ks: int, stride: int, off: int,
                   shift: Optional[torch.Tensor] = None, prelu_in: Optional[torch.Tensor] = None,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """bf16 tensor-core form: conv(prelu_in(x)) * scale + shift with the scale already folded into `w`
    ((Cout, ks*ks*Cin) bf16, tap-major).  The PReLU of a CAB (cod.py:440-442) is applied to the INPUT of its
    second conv while the operand is gathered, so the first conv's epilogue stays a plain store."""
    check_cuda(w, shift, prelu_in)
    _on_cuda(x, out)
    B, h, wd, Cin = x.shape
    Cout, K = w.shape
    assert K == ks * ks * Cin and w.dtype == torch.bfloat16
    oh, ow = out_hw
    M = B * oh * ow
    if out is None:
        out = torch.empty(B, oh, ow, Cout, device=x.device, dtype=torch.float32)
    assert out.shape == (B, oh, ow, Cout)
    col = _col_scratch(x.device, M * K)
    call("dgtd_im2col_act_fwd", x.data_ptr(), _pitch(x), ptr(col), ptr(prelu_in), B, h, wd, Cin, ks, stride, off, oh, ow,
         stream())
    call("dgtd_linear_fwd", ptr(col), ptr(w), ptr(shift), out.data_ptr(), M, Cout, K, _pitch(out), capi.BF16, capi.F32,
         capi.ACT_NONE, stream())
    return out




def conv3_tc(x: torch.Tensor, w: torch.Tensor, shift: Optional[torch.Tensor] = None,
             prelu_in: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """3x3 / stride 1 / pad 1 conv as an implicit tcgen05 GEMM (no im2col in HBM): conv(prelu_in(x)) + shift.
    `w` (Cout, 9 * Cp) bf16 tap-major with the input channels zero-padded to Cp = roundup(Cin, 64)."""
    check_cuda(w, shift, prelu_in)
    _on_cuda(x, out)
    B, h, wd, Cin = x.shape
    Cout = w.shape[0]
    Cp = (Cin + 63) // 64 * 64
    assert w.shape[1] == 9 * Cp and w.dtype == torch.bfloat16
    if out is None:
        out = torch.empty(B, h, wd, Cout, device=x.device, dtype=torch.float32)
    assert out.shape == (B, h, wd, Cout)
    n = B * h * wd * Cp
    from ...model.texture_diffuser import scratch_buffer
    xb = scratch_buffer("hitnet_xb", x.device, n, torch.bfloat16)
    call("dgtd_cast_pad_act_fwd", x.data_ptr(), _pitch(x), ptr(xb), ptr(prelu_in), B * h * wd, Cin, Cp, stream())
    call("dgtd_conv3x3_tc_fwd", ptr(xb), ptr(w), ptr(shift), out.data_ptr(), B, h, wd, Cp, Cout, _pitch(out), stream())
    return out


def channel_sums(x: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Fixed-order partial sums over the pixels of each image: (B, chunks, C), hw."""
    _on_cuda(x)
    B, h, w, C = x.shape
    nch = capi.load().dgtd_channel_sums_chunks(h * w)
    part = torch.empty(B, nch, C, device=x.device, dtype=torch.float32)
    call("dgtd_channel_sums_fwd", x.data_ptr(), _pitch(x), ptr(part), B, h * w, C, stream())
    return part, h * w


def channel_gate(part: torch.Tensor, hw: int, w1: torch.Tensor, w2: torch.Tensor) -> torch.Tensor:
    """sigmoid(W2 relu(W1 mean)) -> (B, Co); W1 (Cr, C), W2 (Co, Cr)."""
    check_cuda(part, w1, w2)
    B, nch, C = part.shape
    Cr, Co = w1.shape[0], w2.shape[0]
    assert w1.shape == (Cr, C) and w2.shape == (Co, Cr)
    gate = torch.empty(B, Co, device=part.device, dtype=torch.float32)
    call("dgtd_channel_gate_fwd", ptr(part), nch, hw, ptr(w1), ptr(w2), ptr(gate), B, C, Cr, Co, stream())
    return gate


def gated_sum(a: torch.Tensor, ga: Optional[torch.Tensor] = None, sa: Optional[torch.Tensor] = None,
              b: Optional[torch.Tensor] = None, gb: Optional[torch.Tensor] = None, sb: Optional[torch.Tensor] = None,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """a * ga[b,c] * sa[b] + b * gb[b,c] * sb[b]."""
    check_cuda(ga, sa, gb, sb)
    _on_cuda(a, b, out)
    B, h, w, C = a.shape
    if out is None:
        out = torch.empty(B, h, w, C, device=a.device, dtype=torch.float32)
    call("dgtd_gated_sum_fwd", a.data_ptr(), _pitch(a), ptr(ga), ptr(sa), b.data_ptr() if b is not None else None,
         _pitch(b) if b is not None else 0, ptr(gb), ptr(sb), out.data_ptr(), _pitch(out), B, h * w, C, stream())
    return out


def resize_ld(x: torch.Tensor, size: Tuple[int, int], align_corners: bool, out: Optional[torch.Tensor] = None):
    _on_cuda(x, out)
    B, h, w, C = x.shape
    if out is None:
        out = torch.empty(B, size[0], size[1], C, device=x.device, dtype=torch.float32)
    assert out.shape == (B, size[0], size[1], C)
    call("dgtd_resize_nhwc_ld_fwd", x.data_ptr(), _pitch(x), out.data_ptr(), _pitch(out), B, h, w, C, size[0], size[1],
         1 if align_corners else 0, stream())
    return out


def copy_channels(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    _on_cuda(x, out)
    assert x.shape == out.shape
    C = x.shape[-1]
    call("dgtd_copy_channels_fwd", x.data_ptr(), _pitch(x), out.data_ptr(), _pitch(out), x.numel() // C, C, stream())
    return out


def head1(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], out: Optional[torch.Tensor] = None,
          accumulate: bool = False) -> torch.Tensor:
    """1-channel 1x1 conv: (B,h,w,C) -> (B,1,h,w) (== (B,h,w) planes)."""
    check_cuda(w, bias, out)
    _on_cuda(x)
    B, h, wd, C = x.shape
    if out is None:
        assert not accumulate
        out = torch.empty(B, 1, h, wd, device=x.device, dtype=torch.float32)
    call("dgtd_head1_fwd", x.data_ptr(), _pitch(x), ptr(w), ptr(bias), ptr(out), B * h * wd, C, 1 if accumulate else 0,
         stream())
    return out


def sigmoid(x: torch.Tensor) -> torch.Tensor:
    check_cuda(x)
    x = x.contiguous()
    out = torch.empty_like(x)
    call("dgtd_sigmoid_fwd", ptr(x), ptr(out), x.numel(), stream())
    return out


def resize_sigmoid_sized(x: torch.Tensor, like: PaddedBatch) -> PaddedBatch:
    """(B,1,h,w) logits -> a PaddedBatch with `like`'s sizes holding per image `sigmoid(resize_nchw(x[b], (H_b,
    W_b)))`, bit for bit (0 in the padding)."""
    check_cuda(x)
    B, C, h, w = x.shape
    assert C == 1 and B == len(like) and x.dtype == torch.float32, (tuple(x.shape), x.dtype, len(like))
    out = like.empty_like()
    _, _, Hmax, Wmax = out.data.shape
    call("dgtd_resize_sigmoid_sized_fwd", ptr(x), ptr(out.data), ptr(out.device_sizes()), B, h, w, Hmax, Wmax,
         stream())
    return out
