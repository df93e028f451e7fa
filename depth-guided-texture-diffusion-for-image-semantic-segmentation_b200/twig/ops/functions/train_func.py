"""Autograd Functions of the training path (trunk + decoders), exact fp32.

Same convention as the reference's ``MSDeformAttnFunction`` (twig/ops/functions/ms_deform_attn_func.py:
19-46): ``forward`` saves what ``backward`` needs, ``backward`` is ``@once_differentiable`` and
returns ``None`` for non-tensor arguments.  All arithmetic runs in ``libdgtd_ops.so``; torch is
used for allocation, views and (in two places) concatenation / slicing copies.
Activations are NHWC fp32.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from .. import capi
from ..capi import ACT_NONE, ACT_RELU, BF16, F32, call, check_cuda, ptr, stream
from . import texture_diffusion_func as OP


def _f32(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return None if t is None else t.detach().contiguous().float()


def _empty(shape, like: torch.Tensor) -> torch.Tensor:
    return torch.empty(shape, device=like.device, dtype=torch.float32)


# ---- primitive wrappers ----------------------------------------------------------------------------
def linear_dgrad(g, w, pre=None, keep=None, gamma=None, rows_per_sample=1, out=None, accumulate=False):
    """dx[M,K] (+)= (keep.gamma.g)[M,N] @ w[N,K] (* gelu'(pre))."""
    N, K = w.shape
    M = g.numel() // N
    dx = _empty((M, K), g) if out is None else out
    call("dgtd_linear_dgrad", ptr(g), ptr(w), ptr(dx), ptr(pre), ptr(keep), ptr(gamma), rows_per_sample, M, N, K,
         int(accumulate), stream())
    return dx


def linear_wgrad(g, a, N, K, keep=None, rows_per_sample=1, conv=None):
    """dw[N,K] = (keep.g)^T @ a; conv = (ks, h, w, Cin, ldx, oh, ow, stride, off) reads `a` through im2col."""
    M = g.numel() // N
    dw = _empty((N, K), g)
    ws = _empty((capi.load().dgtd_linear_wgrad_ws_floats(M, N, K),), g)
    cv = conv if conv is not None else (0, 0, 0, 0, 0, 0, 0, 0, 0)
    call("dgtd_linear_wgrad", ptr(g), a.data_ptr(), ptr(dw), ptr(ws), ptr(keep), rows_per_sample, M, N, K, *cv,
         stream())
    return dw


def colsum(x, N, keep=None, rows_per_sample=1):
    M = x.numel() // N
    ws = _empty(((M + 1023) // 1024 * N,), x)
    out = _empty((N,), x)
    call("dgtd_colsum", ptr(x), ptr(keep), rows_per_sample, ptr(ws), ptr(out), M, N, stream())
    return out


def gelu(x):
    out = torch.empty_like(x)
    call("dgtd_gelu_fwd", ptr(x), ptr(out), x.numel(), stream())
    return out


def ln_rows(x, w, b, eps):
    """LayerNorm over the last dim (fp32), cod.py:1042-1049."""
    return OP.layer_norm(x, w, b, eps, channels_first=False)


def ln_rows_bwd(g, y, w, eps):
    C = y.shape[-1]
    rows = y.numel() // C
    dy = torch.empty_like(y)
    ws = _empty((capi.load().dgtd_ln_rows_bwd_ws_floats(rows, C),), y)
    dw, db = _empty((C,), y), _empty((C,), y)
    call("dgtd_ln_rows_bwd", ptr(g), ptr(y), ptr(w), ptr(dy), ptr(ws), ptr(dw), ptr(db), rows, C, float(eps), stream())
    return dy, dw, db


def dwconv7(x, wT, bias, add=None, flip=False):
    B, h, w, C = x.shape
    y = torch.empty_like(x)
    call("dgtd_dwconv7_fwd", ptr(x), ptr(wT), ptr(bias), ptr(add), ptr(y), B, h, w, C, int(flip), stream())
    return y


def dwconv7_wgrad(x, dy):
    B, h, w, C = x.shape
    ws = _empty(((B * ((h + 7) // 8) + 1) * 50 * C,), x)
    dwT, db = _empty((49, C), x), _empty((C,), x)
    call("dgtd_dwconv7_wgrad", ptr(x), ptr(dy), ptr(ws), ptr(dwT), ptr(db), B, h, w, C, stream())
    return dwT, db


# ---- bf16 / tensor-core helpers (operands of the tcgen05 gradient GEMMs) ------------------------------
def transpose_op(src, mode, aux=None, want_dst=False, want_T=True, keep=None, gamma=None, rows_per_sample=1):
    """One pass over a 2-D tensor producing bf16 `dst` (same layout) and / or `dstT` (transposed):
    mode 0 scale+cast (fp32 src), 1 gelu, 2 src*gelu'(aux), 3 copy (bf16 src).  See dgtd_ops.h."""
    M, N = src.shape
    dst = torch.empty(M, N, device=src.device, dtype=torch.bfloat16) if want_dst else None
    dstT = torch.empty(N, M, device=src.device, dtype=torch.bfloat16) if want_T else None
    call("dgtd_transpose_op", ptr(src), ptr(aux), ptr(dst), ptr(dstT), ptr(keep), ptr(gamma), rows_per_sample, M, N,
         mode, stream())
    return dst, dstT


def eltwise_colsum(src, mode, aux=None, keep=None, rows_per_sample=1):
    """bf16 dst = (mode 0: keep * fp32 src | mode 2: src * gelu'(aux)) AND its fp32 column sums in one pass."""
    M, N = src.shape
    dst = torch.empty(M, N, device=src.device, dtype=torch.bfloat16)
    ws = _empty((capi.load().dgtd_eltwise_colsum_ws_floats(M, N),), src)
    out = torch.empty(N, device=src.device, dtype=torch.float32)
    call("dgtd_eltwise_colsum", ptr(src), ptr(aux), ptr(dst), ptr(keep), rows_per_sample, ptr(ws), ptr(out), M, N, mode,
         stream())
    return dst, out


def wgrad_tc_mn(a, b, transpose_out=False):
    """(Mo x No) = a[Kr,Mo]^T @ b[Kr,No] on tcgen05 (split-K over Kr) straight from row-major bf16 activations
    (column slices allowed: stride(0) = pitch, stride(1) = 1); fp32 result (optionally transposed)."""
    Kr, Mo = a.shape
    No = b.shape[1]
    assert b.shape[0] == Kr and a.stride(1) == 1 and b.stride(1) == 1
    out = _empty((No, Mo) if transpose_out else (Mo, No), a)
    ws = _empty((capi.load().dgtd_wgrad_tc_ws_floats(Mo, No, Kr),), a)
    call("dgtd_wgrad_tc_mn", a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), ptr(out), ptr(ws), Mo, No, Kr,
         int(transpose_out), stream())
    return out


def colsum_bf16(x):
    M, N = x.shape
    ws = _empty(((M + 1023) // 1024 * N,), x)
    out = _empty((N,), x)
    call("dgtd_colsum_bf16", ptr(x), ptr(ws), ptr(out), M, N, stream())
    return out


def ln_rows_any(y, w, b, eps, out_dtype):
    C = y.shape[-1]
    out = torch.empty(y.shape, device=y.device, dtype=torch.bfloat16 if out_dtype == BF16 else torch.float32)
    call("dgtd_ln_rows_fwd", ptr(y), ptr(w), ptr(b), ptr(out), out_dtype, y.numel() // C, C, float(eps), stream())
    return out


def tc_rows_ok(M: int) -> bool:
    """The tcgen05 gradient GEMMs reduce over the M rows: TMA needs 16-byte row pitch, and tiny maps
    are not worth a split-K launch."""
    return M % 8 == 0 and M >= 256


# ---- Functions ---------------------------------------------------------------------------------------
class ConvNextBlockBf16Fn(Function):
    """convnext_Block with bf16 tensor-core GEMMs in forward AND backward (fp32 residual stream,
    fp32 accumulation, fp32 LayerNorm / depthwise conv); same signature as ConvNextBlockFn."""

    @staticmethod
    def forward(ctx, x, dw_w, dw_b, ln_w, ln_b, w1, b1, w2, b2, gamma, keep, eps):
        x = _f32(x)
        B, h, w, C = x.shape
        dwT = _f32(dw_w).reshape(C, 49).t().contiguous()
        dw_b, ln_w, ln_b, w1, b1, w2, b2 = map(_f32, (dw_b, ln_w, ln_b, w1, b1, w2, b2))
        gamma, keep = _f32(gamma), _f32(keep)
        w1b, w2b = w1.to(torch.bfloat16), w2.to(torch.bfloat16)
        y = dwconv7(x, dwT, dw_b)
        a = ln_rows_any(y, ln_w, ln_b, eps, BF16).view(-1, C)
        hpre = OP.linear(a, w1b, b1)                                   # bf16 (M, 4C), pre-activation kept
        hid, _ = transpose_op(hpre, 1, want_dst=True, want_T=False)    # GELU
        out = torch.empty_like(x)
        OP.linear_residual_(hid, w2b, b2, gamma, keep, h * w, x, out=out)
        ctx.eps = eps
        ctx.save_for_backward(x, y, a, hpre, hid, dwT, ln_w, w1b, w2, b2, gamma, keep)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        """Weight gradients read dY and X as they lie in memory (MN-major tcgen05 operands, split over the
        pixel rows): no transposed copies; the layer-scale factor is folded into W2 for the input gradient."""
        x, y, a, hpre, hid, dwT, ln_w, w1b, w2, b2, gamma, keep = ctx.saved_tensors
        g = _f32(g)
        B, h, w, C = x.shape
        rows, C4, M = h * w, 4 * C, B * h * w
        g2 = g.view(M, C)
        gk, s = eltwise_colsum(g2, 0, keep=keep, rows_per_sample=rows)   # bf16 keep*g and its column sums, one pass
        G = wgrad_tc_mn(gk, hid)                                       # (C, 4C) = (keep g)^T hid
        dW2, db2 = torch.empty_like(w2), _empty((C,), g)
        dgamma = _empty((C,), g) if gamma is not None else None
        call("dgtd_layer_scale_finalize", ptr(G), ptr(s), ptr(w2), ptr(b2), ptr(gamma), ptr(dW2), ptr(db2),
             ptr(dgamma), C, C4, stream())
        w2g = w2 if gamma is None else w2 * gamma[:, None]
        dh = OP.linear(gk, w2g.t().to(torch.bfloat16).contiguous(), None)   # bf16 (M, 4C) = (keep g) @ (gamma W2)
        dhpre, db1 = eltwise_colsum(dh, 2, aux=hpre)                   # dH * gelu'(pre) and db1, one pass
        del dh, gk
        dW1 = wgrad_tc_mn(dhpre, a)                                    # (4C, C)
        da = OP.linear(dhpre, w1b.t().contiguous(), None, out_dtype=F32)   # fp32 (M, C)
        del dhpre
        dy, dln_w, dln_b = ln_rows_bwd(da, y, ln_w, ctx.eps)
        dx = dwconv7(dy.view(B, h, w, C), dwT.flip(0).contiguous(), None, add=g)
        ddwT, ddb = dwconv7_wgrad(x, dy.view(B, h, w, C))
        return (dx, ddwT.t().reshape(C, 1, 7, 7), ddb, dln_w, dln_b, dW1, db1, dW2, db2, dgamma, None, None)


class DownsampleBf16Fn(Function):
    """LayerNorm + 2x2/2 conv with the conv (and its gradients) on tcgen05."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, w, b, eps):
        x = _f32(x)
        B, h, wd, C = x.shape
        ln_w, ln_b, b = _f32(ln_w), _f32(ln_b), _f32(b)
        wpb = _f32(w).permute(0, 2, 3, 1).reshape(2 * C, 4 * C).to(torch.bfloat16).contiguous()
        p = OP.ln_patchify(x, ln_w, ln_b, BF16, eps)                   # (M', 4C) bf16
        out = OP.linear(p, wpb, b, out_dtype=F32).view(B, h // 2, wd // 2, 2 * C)
        ctx.eps = eps
        ctx.save_for_backward(x, p, wpb, ln_w)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, p, wpb, ln_w = ctx.saved_tensors
        B, h, wd, C = x.shape
        g = _f32(g)
        g2 = g.view(-1, 2 * C)
        gs, _ = transpose_op(g2, 0, want_dst=True, want_T=False)
        dWp = wgrad_tc_mn(gs, p)                                       # (2C, 4C)
        dW = dWp.view(2 * C, 2, 2, C).permute(0, 3, 1, 2).contiguous()
        db = colsum(g2, 2 * C)
        dp = OP.linear(gs, wpb.t().contiguous(), None, out_dtype=F32)  # (M', 4C) fp32
        da = torch.empty_like(x)
        call("dgtd_unpatchify2", ptr(dp), ptr(da), B, h, wd, C, stream())
        dx, dln_w, dln_b = ln_rows_bwd(da, x, ln_w, ctx.eps)
        return dx, dln_w, dln_b, dW, db, None


class LinearFn(Function):
    """out = a @ w^T + b on (..., K) fp32 rows (head 1x1 convs, cod.py:1160,1174)."""

    @staticmethod
    def forward(ctx, a, w, b):
        a, w2, b = _f32(a), _f32(w).reshape(w.shape[0], -1).contiguous(), _f32(b)
        check_cuda(a, w2, b)
        ctx.wshape = tuple(w.shape)
        ctx.save_for_backward(a, w2)
        return OP.linear(a, w2, b)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        a, w2 = ctx.saved_tensors
        g = _f32(g)
        N, K = w2.shape
        da = linear_dgrad(g, w2).view(a.shape) if ctx.needs_input_grad[0] else None
        dw = linear_wgrad(g, a, N, K).view(ctx.wshape) if ctx.needs_input_grad[1] else None
        db = colsum(g, N) if ctx.needs_input_grad[2] else None
        return da, dw, db


class ConvNextBlockFn(Function):
    """convnext_Block (cod.py:1104-1117) on an NHWC fp32 tensor; out-of-place."""

    @staticmethod
    def forward(ctx, x, dw_w, dw_b, ln_w, ln_b, w1, b1, w2, b2, gamma, keep, eps):
        x = _f32(x)
        B, h, w, C = x.shape
        dwT = _f32(dw_w).reshape(C, 49).t().contiguous()
        dw_b, ln_w, ln_b, w1, b1, w2, b2 = map(_f32, (dw_b, ln_w, ln_b, w1, b1, w2, b2))
        gamma, keep = _f32(gamma), _f32(keep)
        y = dwconv7(x, dwT, dw_b)
        a = ln_rows(y, ln_w, ln_b, eps)
        hpre = OP.linear(a.view(-1, C), w1, b1)
        hid = gelu(hpre)
        out = torch.empty_like(x)
        OP.linear_residual_(hid, w2, b2, gamma, keep, h * w, x, out=out)
        ctx.eps = eps
        ctx.has_gamma = gamma is not None
        ctx.save_for_backward(x, y, a, hpre, dwT, ln_w, w1, w2, b2, gamma, keep)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, y, a, hpre, dwT, ln_w, w1, w2, b2, gamma, keep = ctx.saved_tensors
        g = _f32(g)
        B, h, w, C = x.shape
        rows = h * w
        C4 = 4 * C
        # pwconv2, layer scale, DropPath:  out = x + keep * gamma * (hid @ w2^T + b2)
        s = colsum(g, C, keep, rows)
        hid = gelu(hpre)
        G = linear_wgrad(g, hid, C, C4, keep, rows)
        dW2, db2 = torch.empty_like(w2), _empty((C,), g)
        dgamma = _empty((C,), g) if gamma is not None else None
        call("dgtd_layer_scale_finalize", ptr(G), ptr(s), ptr(w2), ptr(b2), ptr(gamma), ptr(dW2), ptr(db2),
             ptr(dgamma), C, C4, stream())
        del hid, G
        dhpre = linear_dgrad(g, w2, pre=hpre, keep=keep, gamma=gamma, rows_per_sample=rows)   # (M, 4C)
        # pwconv1
        dW1 = linear_wgrad(dhpre, a, C4, C)
        db1 = colsum(dhpre, C4)
        da = linear_dgrad(dhpre, w1)                                                          # (M, C)
        del dhpre
        # LayerNorm, depthwise conv, residual
        dy, dln_w, dln_b = ln_rows_bwd(da, y, ln_w, ctx.eps)
        dx = dwconv7(dy.view(B, h, w, C), dwT.flip(0).contiguous(), None, add=g)   # rotated taps = input gradient
        ddwT, ddb = dwconv7_wgrad(x, dy.view(B, h, w, C))
        return (dx, ddwT.t().reshape(C, 1, 7, 7), ddb, dln_w, dln_b, dW1, db1, dW2, db2, dgamma, None, None)


class StemFn(Function):
    """(bilinear-up(grid) + image) -> conv4x4/4 -> LayerNorm(channels_first): cod.py:1302,1127-1128."""

    @staticmethod
    def forward(ctx, image, grid, w, b, ln_w, ln_b, eps):
        image, grid = _f32(image), _f32(grid)
        B, _, H, W = image.shape
        Cout = w.shape[0]
        w2, b, ln_w, ln_b = _f32(w).reshape(Cout, 48).contiguous(), _f32(b), _f32(ln_w), _f32(ln_b)
        oh, ow = H // 4, W // 4
        patches = _empty((B * oh * ow, 48), image)
        call("dgtd_stem_patchify", ptr(image), ptr(grid), grid.shape[-1] if grid is not None else 0, ptr(patches), F32,
             B, H, W, stream())
        pre = OP.linear(patches, w2, b)
        out = ln_rows(pre, ln_w, ln_b, eps).view(B, oh, ow, Cout)
        ctx.cfg = (B, H, W, Cout, eps, None if grid is None else tuple(grid.shape))
        ctx.save_for_backward(patches, pre, w2, ln_w)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        patches, pre, w2, ln_w = ctx.saved_tensors
        B, H, W, Cout, eps, gshape = ctx.cfg
        g = _f32(g)
        dpre, dln_w, dln_b = ln_rows_bwd(g, pre, ln_w, eps)
        dW = linear_wgrad(dpre, patches, Cout, 48).view(Cout, 3, 4, 4)
        db = colsum(dpre, Cout)
        dgrid = None
        if gshape is not None and ctx.needs_input_grad[1]:
            dpatches = linear_dgrad(dpre, w2)
            dimg = _empty((B, 3, H, W), g)
            call("dgtd_stem_unpatchify", ptr(dpatches), ptr(dimg), B, H, W, stream())
            dgrid = _empty(gshape, g)
            call("dgtd_resize_bilinear_nchw_bwd", ptr(dimg), ptr(dgrid), B * 3, gshape[2], gshape[3], H, W, stream())
        return None, dgrid, dW, db, dln_w, dln_b, None


class DownsampleFn(Function):
    """LayerNorm(channels_first) -> conv 2x2 stride 2 (cod.py:1132-1135) on NHWC."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, w, b, eps):
        x = _f32(x)
        B, h, wd, C = x.shape
        ln_w, ln_b, b = _f32(ln_w), _f32(ln_b), _f32(b)
        wp = _f32(w).permute(0, 2, 3, 1).reshape(2 * C, 4 * C).contiguous()
        a = ln_rows(x, ln_w, ln_b, eps)
        p = _empty((B * (h // 2) * (wd // 2), 4 * C), x)
        call("dgtd_patchify2", ptr(a), ptr(p), B, h, wd, C, stream())
        out = OP.linear(p, wp, b).view(B, h // 2, wd // 2, 2 * C)
        ctx.eps = eps
        ctx.save_for_backward(x, p, wp, ln_w)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, p, wp, ln_w = ctx.saved_tensors
        B, h, wd, C = x.shape
        g = _f32(g)
        dWp = linear_wgrad(g, p, 2 * C, 4 * C)
        dW = dWp.view(2 * C, 2, 2, C).permute(0, 3, 1, 2).contiguous()
        db = colsum(g, 2 * C)
        dp = linear_dgrad(g, wp)
        da = torch.empty_like(x)
        call("dgtd_unpatchify2", ptr(dp), ptr(da), B, h, wd, C, stream())
        dx, dln_w, dln_b = ln_rows_bwd(da, x, ln_w, ctx.eps)
        return dx, dln_w, dln_b, dW, db, None


class FusionFn(Function):
    """bilinear up of the 4 projected levels, concat, 1x1 conv 4C -> C (cod.py:1175-1176)."""

    @staticmethod
    def forward(ctx, l0, l1, l2, l3, wf, bf):
        levels = [_f32(t) for t in (l0, l1, l2, l3)]
        C = wf.shape[0]
        wf2, bf = _f32(wf).reshape(C, 4 * C).contiguous(), _f32(bf)
        B, h0, w0, _ = levels[0].shape
        ups = [levels[0]] + [OP.resize_nhwc(t, (h0, w0)) for t in levels[1:]]
        cat = torch.cat(ups, dim=-1).contiguous()          # data movement only
        out = OP.linear(cat.view(-1, 4 * C), wf2, bf).view(B, h0, w0, C)
        ctx.shapes = [tuple(t.shape) for t in levels]
        ctx.wshape = tuple(wf.shape)
        ctx.save_for_backward(cat, wf2)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        cat, wf2 = ctx.saved_tensors
        g = _f32(g)
        C = wf2.shape[0]
        B, h0, w0, _ = ctx.shapes[0]
        dwf = linear_wgrad(g, cat, C, 4 * C).view(ctx.wshape)
        dbf = colsum(g, C)
        dcat = linear_dgrad(g, wf2).view(B, h0, w0, 4 * C)
        grads = []
        for i, shp in enumerate(ctx.shapes):
            gi = dcat[..., i * C:(i + 1) * C].contiguous()
            if i == 0:
                grads.append(gi)
                continue
            dl = _empty(shp, g)
            call("dgtd_resize_nhwc_bwd", ptr(gi), ptr(dl), B, shp[1], shp[2], C, h0, w0, 0, stream())
            grads.append(dl)
        return grads[0], grads[1], grads[2], grads[3], dwf, dbf


class Conv3x3Fn(Function):
    """3x3 conv, pad 1 (+ReLU) on NHWC fp32 (ShapePropDecoder, cod.py:1217-1221)."""

    @staticmethod
    def forward(ctx, x, w, b, relu):
        x = _f32(x)
        B, h, wd, Cin = x.shape
        Cout = w.shape[0]
        wf = _f32(w)
        wp = wf.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
        out = OP.conv_nhwc(x, wp, _f32(b), Cin, (h, wd), 3, 1, -1, act=ACT_RELU if relu else ACT_NONE)
        # weights of the input-gradient conv: transposed channels, taps rotated by 180 degrees
        wt = wf.flip(2, 3).permute(1, 2, 3, 0).reshape(Cin, 9 * Cout).contiguous()
        ctx.relu = bool(relu)
        ctx.wshape = tuple(w.shape)
        ctx.save_for_backward(x, out if relu else None, wt)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, out, wt = ctx.saved_tensors
        g = _f32(g)
        B, h, wd, Cin = x.shape
        Cout = ctx.wshape[0]
        if ctx.relu:
            gm = torch.empty_like(g)
            call("dgtd_relu_bwd", ptr(g), ptr(out), ptr(gm), g.numel(), stream())
            g = gm
        dx = OP.conv_nhwc(g, wt, None, Cout, (h, wd), 3, 1, -1) if ctx.needs_input_grad[0] else None
        dWp = linear_wgrad(g, x, Cout, 9 * Cin, conv=(3, h, wd, Cin, Cin, h, wd, 1, -1))
        dW = dWp.view(Cout, 3, 3, Cin).permute(0, 3, 1, 2).contiguous()
        db = colsum(g, Cout)
        return dx, dW, db, None


class ResizeNHWCFn(Function):
    """Bilinear resize of an NHWC map (prompt injection, cod.py:1471) with its adjoint."""

    @staticmethod
    def forward(ctx, x, size):
        x = _f32(x)
        ctx.in_shape = tuple(x.shape)
        ctx.size = (int(size[0]), int(size[1]))
        return OP.resize_nhwc(x, ctx.size)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        B, h, w, C = ctx.in_shape
        g = _f32(g)
        dx = _empty(ctx.in_shape, g)
        call("dgtd_resize_nhwc_bwd", ptr(g), ptr(dx), B, h, w, C, ctx.size[0], ctx.size[1], 0, stream())
        return dx, None


class LayerNormRowsFn(Function):
    """LayerNorm over the last dim of an fp32 (..., C) tensor with input / weight / bias gradients (the stand-alone
    differentiable form of the custom `LayerNorm`, cod.py:1025-1049)."""

    @staticmethod
    def forward(ctx, x, w, b, eps):
        x, w, b = _f32(x), _f32(w), _f32(b)
        check_cuda(x, w, b)
        ctx.eps = eps
        ctx.save_for_backward(x, w)
        return ln_rows(x, w, b, eps)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        dx, dw, db = ln_rows_bwd(_f32(g), x, w, ctx.eps)
        return dx, dw, db, None


class LayoutFn(Function):
    """NCHW <-> NHWC copies (pure data movement) with the transposed copy as backward."""

    @staticmethod
    def forward(ctx, x, to_nhwc):
        ctx.to_nhwc = bool(to_nhwc)
        x = _f32(x)
        return OP.nchw_to_nhwc(x) if to_nhwc else OP.nhwc_to_nchw(x)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        g = _f32(g)
        return (OP.nhwc_to_nchw(g) if ctx.to_nhwc else OP.nchw_to_nhwc(g)), None
