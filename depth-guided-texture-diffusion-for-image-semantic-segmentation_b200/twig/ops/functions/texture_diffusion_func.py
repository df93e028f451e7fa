"""Operator functions of the texture-diffusion hot path.

Same role as ``twig/ops/functions/ms_deform_attn_func.py`` in the reference: the Python side
of the native extension.  Every function allocates its outputs with torch (so the caching
allocator and autograd own the memory), passes raw device pointers + the current stream to
``libdgtd_ops.so`` through ctypes and raises ``RuntimeError`` on failure.  Nothing here computes
on the CPU or through ATen kernels.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from .. import capi
from ..capi import ACT_GELU, ACT_NONE, ACT_RELU, BF16, F32, call, check_cuda, ptr, stream

__all__ = [
    "surface_normals", "HighpassPlan", "fft_highpass", "diffusion_front", "MessagePassingFunction",
    "message_passing_core", "message_passing_tiled", "conv1x1_nchw_autograd", "resize_bilinear_nchw_autograd", "conv1x1_nchw", "resize_nchw", "layer_norm",
    "stem", "stem_patches", "ln_rows_", "fusion_sum", "ln_patchify", "dwconv7_ln", "dwconv7_ln_tma", "linear", "linear_ln", "linear_tf32", "linear_residual_", "conv_nhwc", "conv_nhwc_grouped",
    "resize_nhwc", "cast", "nhwc_to_nchw", "nchw_to_nhwc", "enable_gemm_profile", "collect_gemm_profile",
]


# ---- optional per-launch timing of the tensor-core GEMMs (bench.py roofline) --------------------
_PROFILE = {"on": False, "events": []}


def enable_gemm_profile(on: bool = True):
    _PROFILE["on"] = bool(on)
    _PROFILE["events"] = []
    return _PROFILE


def collect_gemm_profile(min_n: int = 0, min_k: int = 0):
    """(total algorithmic FLOPs, total milliseconds, launches) of the profiled tcgen05 GEMMs with
    N >= min_n and K >= min_k."""
    torch.cuda.synchronize()
    ev = [e for e in _PROFILE["events"] if e[3] is None or (e[3][1] >= min_n and e[3][2] >= min_k)]
    flops = sum(e[0] for e in ev)
    ms = sum(e[1].elapsed_time(e[2]) for e in ev)
    return flops, ms, len(ev)


class _timed:
    def __init__(self, flops: float, active: bool, shape=None):
        self.flops, self.active, self.shape = flops, active and _PROFILE["on"], shape

    def __enter__(self):
        if self.active:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.active:
            self.b.record()
            _PROFILE["events"].append((self.flops, self.a, self.b, self.shape))


def _tdtype(code: int) -> torch.dtype:
    return torch.float32 if code == F32 else torch.bfloat16


# ------------------------------------------------------------------------------------------ a1
def surface_normals(depth: torch.Tensor) -> torch.Tensor:
    """cod.py:96-109. depth (B,1,H,W) fp32 -> (B,3,H,W)."""
    check_cuda(depth)
    B, _, H, W = depth.shape
    out = torch.empty(B, 3, H, W, device=depth.device, dtype=torch.float32)
    call("dgtd_surface_normals_fwd", ptr(depth), ptr(out), B, H, W, stream())
    return out


# ------------------------------------------------------------------------------------------ a2
class HighpassPlan:
    """Per-(H,W) constants of the projector form of ``prompt_encoder.fft`` (cod.py:1256-1271)."""

    _cache = {}

    def __init__(self, H: int, W: int, rate: float, device: torch.device):
        line = int((W * H * rate) ** 0.5 // 2)  # cod.py:1261
        self.H, self.W, self.line = H, W, line
        self.Ph = torch.empty(H, H, device=device, dtype=torch.float32)
        self.sc_h = torch.empty(2 * H, device=device, dtype=torch.float32)
        call("dgtd_lowpass_projector", ptr(self.Ph), ptr(self.sc_h), H, line, stream())
        if W == H:
            self.Pw, self.sc_w = self.Ph, self.sc_h
        else:
            self.Pw = torch.empty(W, W, device=device, dtype=torch.float32)
            self.sc_w = torch.empty(2 * W, device=device, dtype=torch.float32)
            call("dgtd_lowpass_projector", ptr(self.Pw), ptr(self.sc_w), W, line, stream())

    @classmethod
    def get(cls, H: int, W: int, rate: float, device: torch.device) -> "HighpassPlan":
        key = (H, W, float(rate), device.index)
        plan = cls._cache.get(key)
        if plan is None:
            plan = cls._cache[key] = cls(H, W, rate, device)
        return plan


def _split_bf16(t: torch.Tensor):
    hi = t.to(torch.bfloat16)
    return hi.contiguous(), (t - hi.float()).to(torch.bfloat16).contiguous()


def fft_highpass(x: torch.Tensor, rate: float = 0.3, tensor_cores: bool = False) -> torch.Tensor:
    """|x - lowpass(x)| per plane, the operator of cod.py:1256-1271.  No gradient (SURVEY 0.7).
    tensor_cores=True: projector products on tcgen05 with a two-term bf16 split (fp32-accurate, ~1e-5)."""
    check_cuda(x)
    assert x.dtype == torch.float32 and x.dim() == 4
    B, C, H, W = x.shape
    plan = HighpassPlan.get(H, W, rate, x.device)
    if tensor_cores and H % 8 == 0 and W % 8 == 0:
        # each split product as one K-concatenated GEMM: [x_hi | x_lo | x_hi] . [P_hi | P_hi | P_lo]^T
        if not hasattr(plan, "tc3"):
            def cat(t):
                hi, lo = _split_bf16(t)
                return torch.cat([hi, hi, lo], 1).contiguous()
            ph = cat(plan.Ph)
            plan.tc3 = (ph, ph if plan.Pw is plan.Ph else cat(plan.Pw))
        ph_cat, pw_cat = plan.tc3
        n = x.numel()
        ws_a = torch.empty(3 * n, device=x.device, dtype=torch.bfloat16)
        ws_f = torch.empty(n, device=x.device, dtype=torch.float32)
        coef = torch.empty(B * C * 4, device=x.device, dtype=torch.float32)
        out = torch.empty_like(x)
        call("dgtd_fft_highpass_tc3_fwd", ptr(x), ptr(ph_cat), ptr(pw_cat), ptr(plan.sc_h), ptr(plan.sc_w), ptr(ws_a),
             ptr(ws_f), ptr(coef), ptr(out), B * C, H, W, stream())
        return out
    tmp = torch.empty_like(x)
    coef = torch.empty(B * C * 4, device=x.device, dtype=torch.float32)
    out = torch.empty_like(x)
    call("dgtd_fft_highpass_fwd", ptr(x), ptr(plan.Ph), ptr(plan.Pw), ptr(plan.sc_h), ptr(plan.sc_w),
         ptr(tmp), ptr(coef), ptr(out), B * C, H, W, stream())
    return out


# ------------------------------------------------------------------------------------------ a3..a6
def diffusion_front(emb1: torch.Tensor, depth: torch.Tensor, reg_w, reg_b, enc_w, enc_b, conv_w, conv_b,
                    grid: int = 12, steps: int = 4, save_wn: bool = False):
    """Fused cod.py:1295-1298 + :1201-1206 -> (B,3,G,G); also returns the saved states
    (B,T+1,C,G,G) and, on request, the normalised weights (B,C,49,G*G)."""
    check_cuda(emb1, depth, reg_w, reg_b, enc_w, enc_b, conv_w, conv_b)
    B, _, H, W = emb1.shape
    C = enc_w.shape[0]
    out = torch.empty(B, 3, grid, grid, device=emb1.device, dtype=torch.float32)
    states = torch.empty(B, steps + 1, C, grid, grid, device=emb1.device, dtype=torch.float32)
    wn = torch.empty(B, C, 49, grid * grid, device=emb1.device, dtype=torch.float32) if save_wn else None
    call("dgtd_diffusion_front_fwd", ptr(emb1), ptr(depth), ptr(reg_w), ptr(reg_b), ptr(enc_w), ptr(enc_b),
         ptr(conv_w), ptr(conv_b), ptr(out), ptr(states), ptr(wn), B, H, W, grid, C, steps, stream())
    return out, states, wn


class MessagePassingFunction(Function):
    """The diffusion core of ``MessagePassing.forward`` (cod.py:1190-1205) with its backward."""

    @staticmethod
    def forward(ctx, x: torch.Tensor, weight: torch.Tensor, steps: int, eps: float):
        x = x.contiguous().float()
        weight = weight.contiguous().float()
        check_cuda(x, weight)
        n, c, h, w = x.shape
        wc = weight.shape[1] // 49
        out = torch.empty_like(x)
        need_grad = x.requires_grad or weight.requires_grad
        states = torch.empty(n, steps + 1, c, h, w, device=x.device, dtype=torch.float32) if need_grad else None
        call("dgtd_message_passing_fwd", ptr(x), ptr(weight), ptr(out), ptr(states), n, c, h, w, wc, steps,
             float(eps), stream())
        if need_grad:
            ctx.save_for_backward(weight, states)
        ctx.cfg = (n, c, h, w, wc, steps, float(eps))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        weight, states = ctx.saved_tensors
        n, c, h, w, wc, steps, eps = ctx.cfg
        grad_out = grad_out.contiguous().float()
        gx = torch.empty(n, c, h, w, device=grad_out.device, dtype=torch.float32)
        gw = torch.empty_like(weight)
        call("dgtd_message_passing_bwd", ptr(grad_out), ptr(weight), ptr(states), ptr(gx), ptr(gw), n, c, h,
             w, wc, steps, eps, stream())
        return gx, gw, None, None


def message_passing_core(x: torch.Tensor, weight: torch.Tensor, steps: int = 4, eps: float = 1e-5):
    return MessagePassingFunction.apply(x, weight, steps, eps)


class Conv1x1NCHWFunction(Function):
    """1x1 conv (+ optional sigmoid) on NCHW maps with gradients for x, weight and bias:
    ShapePropWeightRegressor (cod.py:1058-1060), encoder1 (:1297), message_passing.conv (:1206)."""

    @staticmethod
    def forward(ctx, x, weight, bias, sigmoid: bool):
        x = x.contiguous().float()
        w2 = weight.reshape(weight.shape[0], -1).contiguous().float()
        out = conv1x1_nchw(x, w2, None if bias is None else bias.contiguous().float(), sigmoid)
        ctx.sigmoid = bool(sigmoid)
        ctx.wshape = tuple(weight.shape)
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, w2, out if sigmoid else None)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, w2, y = ctx.saved_tensors
        g = g.contiguous().float()
        B, Cin = x.shape[0], x.shape[1]
        HW = x.numel() // (B * Cin)
        Cout = w2.shape[0]
        gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gw = torch.empty_like(w2) if (ctx.needs_input_grad[1] or ctx.needs_input_grad[2]) else None
        gb = torch.empty(Cout, device=x.device, dtype=torch.float32) if gw is not None else None
        call("dgtd_conv1x1_nchw_bwd", ptr(g), ptr(y), ptr(x), ptr(w2), ptr(gx), ptr(gw), ptr(gb), B, Cin, Cout, HW,
             stream())
        return (gx, gw.reshape(ctx.wshape) if gw is not None and ctx.needs_input_grad[1] else None,
                gb if ctx.has_bias and ctx.needs_input_grad[2] else None, None)


class ResizeBilinearNCHWFunction(Function):
    """F.interpolate(mode='bilinear', align_corners=False) with its exact adjoint (cod.py:1207,1298)."""

    @staticmethod
    def forward(ctx, x, size):
        x = x.contiguous().float()
        ctx.in_hw = (x.shape[2], x.shape[3])
        ctx.out_hw = (int(size[0]), int(size[1]))
        return resize_nchw(x, ctx.out_hw, bilinear=True)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        g = g.contiguous().float()
        B, C = g.shape[0], g.shape[1]
        gx = torch.empty(B, C, ctx.in_hw[0], ctx.in_hw[1], device=g.device, dtype=torch.float32)
        call("dgtd_resize_bilinear_nchw_bwd", ptr(g), ptr(gx), B * C, ctx.in_hw[0], ctx.in_hw[1], ctx.out_hw[0],
             ctx.out_hw[1], stream())
        return gx, None


def conv1x1_nchw_autograd(x, weight, bias, sigmoid: bool = False):
    return Conv1x1NCHWFunction.apply(x, weight, bias, sigmoid)


def resize_bilinear_nchw_autograd(x, size):
    return ResizeBilinearNCHWFunction.apply(x, size)


def message_passing_tiled(x: torch.Tensor, weight: torch.Tensor, steps: int, eps: float = 1e-5, impl: str = "auto"):
    """Large-map variant: x (n,h,w,c) channels-last storage (fp32|bf16), weight (n,49,h,w) fp32.
    impl: "auto" (tensor-pipe banded GEMM when the shape qualifies, else the SIMT kernel), "simt", "tc"."""
    check_cuda(x, weight)
    n, h, w, c = x.shape
    out = torch.empty_like(x)
    tmp = torch.empty_like(x) if steps > 1 else None
    if impl == "tc":
        call("dgtd_message_passing_tc_fwd", ptr(x), ptr(weight), ptr(out), ptr(tmp), n, h, w, c, steps,
             float(eps), capi.dtype_code(x.dtype), stream())
        return out
    assert impl in ("auto", "simt")
    call("dgtd_message_passing_tiled_fwd" if impl == "auto" else "dgtd_message_passing_tiled_simt_fwd", ptr(x),
         ptr(weight), ptr(out), ptr(tmp), n, h, w, c, steps, float(eps), capi.dtype_code(x.dtype), stream())
    return out


def message_passing_regress(x: torch.Tensor, guide: torch.Tensor, reg_w: torch.Tensor, reg_b: torch.Tensor,
                            steps: int, eps: float = 1e-5, fast_sigmoid: bool = False) -> torch.Tensor:
    """Large-map variant with the model's per-channel weights generated on chip: x (n,h,w,c) channels-last
    storage (fp32|bf16), guide (n,3,h,w) fp32, reg_w (c*49,3[,1,1]), reg_b (c*49) -- the
    ShapePropWeightRegressor parameters (cod.py:1051-1060)."""
    check_cuda(x, guide, reg_w, reg_b)
    n, h, w, c = x.shape
    assert guide.shape == (n, 3, h, w) and reg_w.numel() == c * 49 * 3 and reg_b.numel() == c * 49
    packed = torch.empty(c * 49, 4, device=x.device, dtype=torch.float32)
    call("dgtd_pack_regressor", ptr(reg_w.detach().reshape(c * 49, 3).float().contiguous()),
         ptr(reg_b.detach().float().contiguous()), ptr(packed), c, stream())
    out = torch.empty_like(x)
    tmp = torch.empty_like(x) if steps > 1 else None
    call("dgtd_message_passing_regress_fwd", ptr(x), ptr(guide.contiguous().float()), ptr(packed), ptr(out), ptr(tmp),
         n, h, w, c, steps, float(eps), capi.dtype_code(x.dtype), int(fast_sigmoid), stream())
    return out


# ------------------------------------------------------------------------------------------ helpers
def conv1x1_nchw(x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], sigmoid: bool = False):
    check_cuda(x, w, b)
    B, Cin = x.shape[0], x.shape[1]
    HW = x.numel() // (B * Cin)
    Cout = w.shape[0]
    out = torch.empty((B, Cout) + tuple(x.shape[2:]), device=x.device, dtype=torch.float32)
    call("dgtd_conv1x1_nchw_fwd", ptr(x), ptr(w), ptr(b), ptr(out), B, Cin, Cout, HW, int(sigmoid), stream())
    return out


def resize_nchw(x: torch.Tensor, size: Sequence[int], bilinear: bool = True) -> torch.Tensor:
    check_cuda(x)
    B, C, h, w = x.shape
    oh, ow = int(size[0]), int(size[1])
    out = torch.empty(B, C, oh, ow, device=x.device, dtype=torch.float32)
    call("dgtd_resize_nchw_fwd", ptr(x), ptr(out), B * C, h, w, oh, ow, int(bilinear), stream())
    return out


def layer_norm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float, channels_first: bool):
    check_cuda(x, w, b)
    out = torch.empty_like(x)
    if channels_first:
        outer, C = x.shape[0], x.shape[1]
        inner = x.numel() // (outer * C)
    else:
        C = x.shape[-1]
        outer, inner = x.numel() // C, 1
    call("dgtd_layer_norm_fwd", ptr(x), ptr(w), ptr(b), ptr(out), outer, C, inner, float(eps), stream())
    return out


# ------------------------------------------------------------------------------------------ a7/a8
def stem(image: torch.Tensor, grid: Optional[torch.Tensor], w, b, ln_w, ln_b, eps: float = 1e-6):
    """(up(grid)+image) -> conv4x4/4 -> LN : returns NHWC (B,H/4,W/4,Cout) fp32."""
    check_cuda(image, grid, w, b, ln_w, ln_b)
    B, _, H, W = image.shape
    Cout = w.shape[0]
    out = torch.empty(B, H // 4, W // 4, Cout, device=image.device, dtype=torch.float32)
    G = grid.shape[-1] if grid is not None else 0
    call("dgtd_stem_fwd", ptr(image), ptr(grid), G, ptr(w), ptr(b), ptr(ln_w), ptr(ln_b), ptr(out), B, H, W,
         Cout, float(eps), stream())
    return out


def ln_patchify(x: torch.Tensor, ln_w, ln_b, out_dtype: int, eps: float = 1e-6) -> torch.Tensor:
    """x NHWC (B,h,w,C) fp32 -> (B*(h//2)*(w//2), 4C) rows ordered (dy,dx,c)."""
    check_cuda(x, ln_w, ln_b)
    B, h, w, C = x.shape
    out = torch.empty(B * (h // 2) * (w // 2), 4 * C, device=x.device, dtype=_tdtype(out_dtype))
    call("dgtd_ln_patchify_fwd", ptr(x), ptr(ln_w), ptr(ln_b), ptr(out), out_dtype, B, h, w, C, float(eps),
         stream())
    return out


def dwconv7_ln(x: torch.Tensor, dw_w, dw_b, ln_w, ln_b, out_dtype: int, eps: float = 1e-6) -> torch.Tensor:
    check_cuda(x, dw_w, dw_b, ln_w, ln_b)
    B, h, w, C = x.shape
    out = torch.empty(B, h, w, C, device=x.device, dtype=_tdtype(out_dtype))
    call("dgtd_dwconv7_ln_fwd", ptr(x), ptr(dw_w), ptr(dw_b), ptr(ln_w), ptr(ln_b), ptr(out), out_dtype, B, h,
         w, C, float(eps), stream())
    return out


def dwconv7_ln_tma(x: torch.Tensor, dw_wT, dw_b, ln_w, ln_b, out_dtype: int, ws: torch.Tensor,
                   eps: float = 1e-6) -> torch.Tensor:
    """TMA-staged variant for large maps: dw_wT is (49, C); ws is a (B,h,w,C) fp32 scratch."""
    check_cuda(x, dw_wT, dw_b, ln_w, ln_b, ws)
    B, h, w, C = x.shape
    assert ws.numel() >= x.numel() and ws.dtype == torch.float32
    out = torch.empty(B, h, w, C, device=x.device, dtype=_tdtype(out_dtype))
    call("dgtd_dwconv7_ln_tma_fwd", ptr(x), ptr(dw_wT), ptr(dw_b), ptr(ln_w), ptr(ln_b), ptr(ws), ptr(out),
         out_dtype, B, h, w, C, float(eps), stream())
    return out


def dwconv7_stats_tma(x: torch.Tensor, dw_wT, dw_b, eps: float = 1e-6):
    """bf16-mode block front with the LayerNorm folded into pwconv1: returns (y bf16 (B,h,w,C) = depthwise 7x7 of x,
    stats (B*h*w, 2) fp32 = (mean, rstd) per pixel of the stored values)."""
    check_cuda(x, dw_wT, dw_b)
    B, h, w, C = x.shape
    y = torch.empty(B, h, w, C, device=x.device, dtype=torch.bfloat16)
    stats = torch.empty(B * h * w, 2, device=x.device, dtype=torch.float32)
    call("dgtd_dwconv7_stats_tma_fwd", ptr(x), ptr(dw_wT), ptr(dw_b), ptr(y), ptr(stats), B, h, w, C, float(eps), stream())
    return y, stats


def linear_lnfold(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, col_s: torch.Tensor, row_stats: torch.Tensor,
                  act: int = ACT_NONE, out_dtype: int = BF16) -> torch.Tensor:
    """act(LN(a) @ W1^T + b1) with the LayerNorm applied in the GEMM epilogue (see dgtd_linear_lnfold_fwd)."""
    check_cuda(a, w, bias, col_s, row_stats)
    K = a.shape[-1]
    M = a.numel() // K
    N = w.shape[0]
    assert w.shape[1] == K and a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and row_stats.shape == (M, 2)
    out = torch.empty(tuple(a.shape[:-1]) + (N,), device=a.device, dtype=_tdtype(out_dtype))
    with _timed(2.0 * M * N * K, True, (M, N, K)):
        call("dgtd_linear_lnfold_fwd", ptr(a), ptr(w), ptr(bias), ptr(col_s), ptr(row_stats), ptr(out), M, N, K, N,
             out_dtype, act, stream())
    return out


def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], act: int = ACT_NONE,
           out_dtype: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[M,N] = act(a[M,K] @ w[N,K]^T + bias).  a and w share a dtype (fp32 exact / bf16 tcgen05)."""
    check_cuda(a, w, bias)
    K = a.shape[-1]
    M = a.numel() // K
    N = w.shape[0]
    assert w.shape[1] == K and a.dtype == w.dtype
    din = capi.dtype_code(a.dtype)
    dout = din if out_dtype is None else out_dtype
    if out is None:
        out = torch.empty(tuple(a.shape[:-1]) + (N,), device=a.device, dtype=_tdtype(dout))
    ldo = out.shape[-1]
    with _timed(2.0 * M * N * K, din == BF16, (M, N, K)):
        call("dgtd_linear_fwd", ptr(a), ptr(w), ptr(bias), ptr(out), M, N, K, ldo, din, dout, act, stream())
    return out


def linear_ln(a: torch.Tensor, w: torch.Tensor, bias, ln_w: torch.Tensor, ln_b: torch.Tensor, eps: float) -> torch.Tensor:
    """out[M,128] fp32 = LayerNorm_rows(a[M,K] bf16 @ w[128,K]^T bf16 + bias) * ln_w + ln_b, the LayerNorm fused in the GEMM's
    epilogue (M >= 256)."""
    check_cuda(a, w, bias, ln_w, ln_b)
    K = a.shape[-1]
    M = a.numel() // K
    N = w.shape[0]
    assert w.shape[1] == K and a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.is_contiguous()
    out = torch.empty(tuple(a.shape[:-1]) + (N,), device=a.device, dtype=torch.float32)
    call("dgtd_linear_ln_fwd", ptr(a), ptr(w), ptr(bias), ptr(ln_w), ptr(ln_b), float(eps), ptr(out), M, N, K, stream())
    return out


def linear_tf32(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """out[M,N] fp32 = a[M,K] fp32 @ w[N,K]^T fp32 + bias on tcgen05 kind::tf32 (N <= 64): a thin projection of an fp32
    activation without the bf16 copy of `linear`."""
    check_cuda(a, w, bias)
    K = a.shape[-1]
    M = a.numel() // K
    N = w.shape[0]
    assert w.shape[1] == K and a.dtype == torch.float32 and w.dtype == torch.float32 and a.is_contiguous()
    out = torch.empty(tuple(a.shape[:-1]) + (N,), device=a.device, dtype=torch.float32)
    call("dgtd_linear_tf32_fwd", ptr(a), ptr(w), ptr(bias), ptr(out), M, N, K, N, stream())
    return out


def linear_residual_(a: torch.Tensor, w: torch.Tensor, bias, gamma, keep: Optional[torch.Tensor],
                     rows_per_sample: int, residual: torch.Tensor, out: Optional[torch.Tensor] = None):
    """out = residual + keep[m//rows] * gamma * (a @ w^T + bias); in place on `residual` when
    `out` is None (each element is read and written by the same thread)."""
    check_cuda(a, w, bias, gamma, keep, residual)
    K = a.shape[-1]
    M = a.numel() // K
    N = w.shape[0]
    assert residual.dtype == torch.float32 and residual.numel() == M * N
    out = residual if out is None else out
    with _timed(2.0 * M * N * K, a.dtype == torch.bfloat16, (M, N, K)):
        call("dgtd_linear_residual_fwd", ptr(a), ptr(w), ptr(bias), ptr(gamma), ptr(keep), rows_per_sample,
             ptr(residual), ptr(out), M, N, K, capi.dtype_code(a.dtype), stream())
    return out


MLP_FUSED_C = (128,)   # channel counts dgtd_convnext_mlp_fused_fwd is built for


def convnext_mlp_fused_(y: torch.Tensor, row_stats: torch.Tensor, w1: torch.Tensor, col_s: torch.Tensor,
                        cbias: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, gamma: Optional[torch.Tensor],
                        residual: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = residual + gamma * (GELU(LN(y) @ W1^T + b1) @ W2^T + b2) in one kernel (hidden tensor on chip); in place on
    `residual` when `out` is None.  y (M, C) bf16 conv output, row_stats (M, 2), w1 (4C, C) bf16 = W1 * ln_weight,
    w2 (C, 4C) bf16."""
    check_cuda(y, row_stats, w1, col_s, cbias, w2, b2, gamma, residual)
    C = y.shape[-1]
    M = y.numel() // C
    assert y.dtype == torch.bfloat16 and w1.dtype == torch.bfloat16 and w2.dtype == torch.bfloat16
    assert w1.shape == (4 * C, C) and w2.shape == (C, 4 * C) and row_stats.shape == (M, 2)
    assert residual.dtype == torch.float32 and residual.numel() == M * C
    out = residual if out is None else out
    with _timed(4.0 * M * C * 4 * C, True, (M, 4 * C, C)):
        call("dgtd_convnext_mlp_fused_fwd", ptr(y), ptr(row_stats), ptr(w1), ptr(col_s), ptr(cbias), ptr(w2), ptr(b2),
             ptr(gamma), ptr(residual), ptr(out), M, C, stream())
    return out


# ------------------------------------------------------------------------------------------ a9
def fusion_sum(levels: List[torch.Tensor], hw: List[Tuple[int, int]], bias, B: int, want_nhwc=True,
               want_nchw=False, pad_to: int = 0):
    """levels[i]: (B*h_i*w_i, C) fp32 with the fusion conv already folded in; out = bias + sum_i up(levels[i]).
    Returns (nhwc, nchw, padded-bf16) tensors."""
    check_cuda(*levels, bias)
    C = levels[0].shape[-1]
    dev = levels[0].device
    h0, w0 = hw[0]
    nhwc = torch.empty(B, h0, w0, C, device=dev, dtype=torch.float32) if want_nhwc else None
    nchw = torch.empty(B, C, h0, w0, device=dev, dtype=torch.float32) if want_nchw else None
    pad = torch.empty(B, h0, w0, pad_to, device=dev, dtype=torch.bfloat16) if pad_to else None
    hw_arr = (capi.c_int * 8)(*[v for pair in hw for v in pair])
    call("dgtd_fusion_sum_fwd", ptr(levels[0]), ptr(levels[1]), ptr(levels[2]), ptr(levels[3]), hw_arr,
         ptr(bias), ptr(nhwc), ptr(nchw), ptr(pad), pad_to, B, C, stream())
    return nhwc, nchw, pad


def stem_patches(image: torch.Tensor, grid: Optional[torch.Tensor], out_dtype: int) -> torch.Tensor:
    """(up(grid)+image) gathered as 4x4/4 patches: (B*(H/4)*(W/4), 48) rows ordered (ci,ky,kx)."""
    check_cuda(image, grid)
    B, _, H, W = image.shape
    out = torch.empty(B * (H // 4) * (W // 4), 48, device=image.device, dtype=_tdtype(out_dtype))
    call("dgtd_stem_patchify", ptr(image), ptr(grid), grid.shape[-1] if grid is not None else 0, ptr(out), out_dtype,
         B, H, W, stream())
    return out


def ln_rows_(y: torch.Tensor, ln_w, ln_b, eps: float = 1e-6) -> torch.Tensor:
    """In-place LayerNorm over the last dim of an fp32 tensor (each row is read into registers before it is
    written); C a multiple of 128."""
    check_cuda(y, ln_w, ln_b)
    C = y.shape[-1]
    call("dgtd_ln_rows_fwd", ptr(y), ptr(ln_w), ptr(ln_b), ptr(y), F32, y.numel() // C, C, float(eps), stream())
    return y


# ------------------------------------------------------------------------------------------ a10/a11
def conv_nhwc(x: torch.Tensor, w: torch.Tensor, bias, Cin: int, out_hw: Tuple[int, int], ks: int,
              stride: int, off: int, act: int = ACT_NONE, out: Optional[torch.Tensor] = None,
              out_dtype: Optional[int] = None, Cout: Optional[int] = None) -> torch.Tensor:
    """KxK conv over NHWC as implicit GEMM.  `x` may be a channel slice of a wider tensor
    (last-dim stride 1, pixel stride = ldx); `w` is packed (Cout, ks*ks*Cin) tap-major."""
    B, h, wd = x.shape[0], x.shape[1], x.shape[2]
    ldx = x.stride(2)
    assert x.stride(3) == 1 and x.stride(1) == wd * ldx and x.stride(0) == h * wd * ldx
    Cout = w.shape[0] if Cout is None else Cout
    oh, ow = out_hw
    din = capi.dtype_code(x.dtype)
    dout = din if out_dtype is None else out_dtype
    if out is None:
        out = torch.empty(B, oh, ow, Cout, device=x.device, dtype=_tdtype(dout))
    ldo = out.stride(2)
    call("dgtd_conv_nhwc_fwd", x.data_ptr(), ptr(w), ptr(bias), out.data_ptr(), B, h, wd, Cin, ldx, oh, ow,
         Cout, ldo, ks, stride, off, act, din, dout, stream())
    return out


def conv_nhwc_grouped(x: torch.Tensor, w: torch.Tensor, bias, Cin: int, out_hw: Tuple[int, int], ks: int,
                      stride: int, off: int, act: int, out: torch.Tensor, Cout: int, ldo: int, groups: int,
                      x_group_stride: int, w_group_rows: int, out_group_stride: int) -> torch.Tensor:
    """Grouped implicit-GEMM conv (all decoders of a stage in one launch); see dgtd_ops.h."""
    B, h, wd = x.shape[0], x.shape[1], x.shape[2]
    ldx = x.stride(2)
    assert x.stride(3) == 1 and x.stride(1) == wd * ldx and x.stride(0) == h * wd * ldx
    oh, ow = out_hw
    call("dgtd_conv_nhwc_grouped_fwd", x.data_ptr(), ptr(w), ptr(bias), out.data_ptr(), B, h, wd, Cin, ldx,
         oh, ow, Cout, ldo, ks, stride, off, act, capi.dtype_code(x.dtype), capi.dtype_code(out.dtype), groups,
         x_group_stride, w_group_rows, out_group_stride, stream())
    return out


def resize_nhwc(x: torch.Tensor, size: Tuple[int, int], out_dtype: Optional[int] = None) -> torch.Tensor:
    check_cuda(x)
    B, h, w, C = x.shape
    din = capi.dtype_code(x.dtype)
    dout = din if out_dtype is None else out_dtype
    out = torch.empty(B, size[0], size[1], C, device=x.device, dtype=_tdtype(dout))
    call("dgtd_resize_nhwc_fwd", ptr(x), ptr(out), B, h, w, C, size[0], size[1], din, dout, stream())
    return out


# ------------------------------------------------------------------------------------------ plumbing
def cast(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    check_cuda(x)
    out = torch.empty(x.shape, device=x.device, dtype=dtype)
    call("dgtd_cast_fwd", ptr(x), ptr(out), x.numel(), capi.dtype_code(x.dtype), capi.dtype_code(dtype),
         stream())
    return out


def nhwc_to_nchw(x: torch.Tensor, C: Optional[int] = None) -> torch.Tensor:
    check_cuda(x)
    B, h, w, ld = x.shape
    C = ld if C is None else C
    out = torch.empty(B, C, h, w, device=x.device, dtype=torch.float32)
    call("dgtd_nhwc_to_nchw_fwd", ptr(x), ptr(out), B, h, w, C, ld, capi.dtype_code(x.dtype), stream())
    return out


def nchw_to_nhwc(x: torch.Tensor, dtype: torch.dtype = torch.float32, ld: Optional[int] = None):
    check_cuda(x)
    B, C, h, w = x.shape
    ld = C if ld is None else ld
    out = torch.empty(B, h, w, ld, device=x.device, dtype=dtype)
    call("dgtd_nchw_to_nhwc_fwd", ptr(x), ptr(out), B, h, w, C, ld, capi.dtype_code(dtype), stream())
    return out
