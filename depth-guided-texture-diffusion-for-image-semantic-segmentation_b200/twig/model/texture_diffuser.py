"""`nn.Module` mirror of the texture diffuser, ``twig/model/cod.py:1025-1323`` in the reference.

Same class names, constructor / forward signatures, attribute names (hence identical
``state_dict`` keys and YAML ``custom_keys`` prefixes, config/cod.yml:88-101) and the same
parameter initialisation order, so a reference checkpoint loads unchanged and
``torch.manual_seed(s)`` + construction gives bit-identical parameters.  Every ``forward`` runs on
the sm_100a kernels of ``libdgtd_ops.so``; there is no ATen compute path and no CPU fallback.

Precision: fp32 (exact CUDA-core path) by default; bf16 operands on tcgen05 tensor cores with
fp32 accumulation / fp32 residual stream when ``set_precision(module, "bf16")`` was called or the
forward runs under ``torch.autocast``.
"""
from __future__ import annotations

import os

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from ..ops.capi import ACT_GELU, ACT_NONE, ACT_RELU, BF16, F32
from ..ops.functions import texture_diffusion_func as OP
from ..ops.functions import train_func as TF
from ..ops.functions import decoder_bank as DB

__all__ = [
    "LayerNorm", "ShapePropWeightRegressor", "convnext_Block", "ShapePropEncoder", "MessagePassing",
    "ShapePropDecoder", "prompt_encoder", "prompt_decoder", "DropPath", "init_weights_", "set_precision",
    "build_texture_diffuser", "pvt_token_grids", "texture_prompts", "texture_prompts_train", "PVT_EMBED_DIMS",
    "PVT_DEPTHS",
]

# bf16 inference: fold each block's LayerNorm into pwconv1 (no normalised copy, no fp32 conv scratch).  The folded form
# centres in fp32 AFTER the bf16 rounding of the un-normalised conv output, i.e. it loses accuracy when a pixel's
# channel mean dwarfs its channel spread (|mean| >> std); DGTD_LN_FOLD=0 keeps the two-pass form.
LN_FOLD = os.environ.get("DGTD_LN_FOLD", "1") != "0"

PVT_EMBED_DIMS = (64, 128, 320, 512)  # pvt_v2_b2, cod.py:1785
PVT_DEPTHS = (3, 4, 6, 3)             # cod.py:1786


# ------------------------------------------------------------------------------------------------
def _mode(module: nn.Module) -> int:
    p = getattr(module, "_dgtd_precision", None)
    if p is None:
        p = "bf16" if torch.is_autocast_enabled() else "fp32"
    return BF16 if p == "bf16" else F32


def set_precision(module: nn.Module, precision: Optional[str]) -> nn.Module:
    """precision in {"fp32", "bf16", None}; None = follow torch.autocast."""
    assert precision in ("fp32", "bf16", None)
    for m in module.modules():
        m._dgtd_precision = precision
    return module


class _Packed:
    """Cache of re-laid-out / down-cast parameters, refreshed when the source changes
    (``load_state_dict`` and optimizer steps bump ``Tensor._version``)."""

    def __init__(self):
        self._store: Dict[str, Tuple[tuple, torch.Tensor]] = {}

    def get(self, key: str, srcs: Sequence[torch.Tensor], fn):
        sig = tuple((t.data_ptr(), t._version, t.device) for t in srcs)
        hit = self._store.get(key)
        if hit is not None and hit[0] == sig:
            return hit[1]
        with torch.no_grad():
            val = fn()
            if hit is not None and _refresh_in_place(hit[1], val):
                # same shapes as before: overwrite the old shadow instead of replacing it, so that a captured CUDA
                # graph that reads the shadow's storage (twig/graphs.py::GraphedPredict) sees the new weights and
                # never a freed block
                val = hit[1]
        self._store[key] = (sig, val)
        return val


def _refresh_in_place(old, new) -> bool:
    if isinstance(old, torch.Tensor) and isinstance(new, torch.Tensor):
        if old.shape != new.shape or old.dtype != new.dtype or old.device != new.device:
            return False
        if old.data_ptr() != new.data_ptr():
            old.copy_(new)
        return True
    if isinstance(old, (tuple, list)) and isinstance(new, (tuple, list)) and len(old) == len(new):
        ok = all(isinstance(a, torch.Tensor) and isinstance(b, torch.Tensor) and a.shape == b.shape and a.dtype == b.dtype
                 and a.device == b.device for a, b in zip(old, new))
        if not ok:
            return False
        for a, b in zip(old, new):
            if a.data_ptr() != b.data_ptr():
                a.copy_(b)
        return True
    return False


def _packed(module: nn.Module) -> _Packed:
    pk = module.__dict__.get("_dgtd_packed")
    if pk is None:
        pk = module.__dict__["_dgtd_packed"] = _Packed()
    return pk


_SCRATCH: Dict[tuple, torch.Tensor] = {}


def scratch_buffer(name: str, device: torch.device, numel: int, dtype: torch.dtype) -> torch.Tensor:
    """Scratch reused by consecutive launches of one call (producer and consumer are stream-ordered).

    * eager: a grow-only buffer per (name, device, stream) -- two streams never share one, and growing only drops
      the old block back to the stream-ordered caching allocator;
    * under CUDA-graph capture: a fresh allocation from the capturing graph's private pool, never cached, so no
      eager call can later replace or free memory a captured graph writes to (ADVICE r1)."""
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(numel, device=device, dtype=dtype)
    key = (name, device, torch.cuda.current_stream(device).cuda_stream, dtype)
    buf = _SCRATCH.get(key)
    if buf is None or buf.numel() < numel:
        buf = _SCRATCH[key] = torch.empty(numel, device=device, dtype=dtype)
    return buf


def _scratch(device: torch.device, numel: int) -> torch.Tensor:
    """fp32 scratch of the ConvNeXt blocks."""
    return scratch_buffer("block", device, numel, torch.float32)


def _as(t: torch.Tensor, mode: int) -> torch.Tensor:
    return t.detach().to(torch.bfloat16).contiguous() if mode == BF16 else t.detach().float().contiguous()


def _wants_grad(module: nn.Module, *inputs) -> bool:
    """True when the forward has to build an autograd graph (training path: exact fp32
    autograd Functions, ops/functions/train_func.py); False = fused inference kernels."""
    if not torch.is_grad_enabled():
        return False
    return any(p.requires_grad for p in module.parameters()) or any(
        isinstance(t, torch.Tensor) and t.requires_grad for t in inputs)


# ------------------------------------------------------------------------------------------------
class DropPath(nn.Module):
    """timm ``DropPath`` (per-sample stochastic depth, scale by 1/keep_prob); cod.py:816,1102."""

    def __init__(self, drop_prob: float = 0.0, scale_by_keep: bool = True):
        super().__init__()
        self.drop_prob = drop_prob
        self.scale_by_keep = scale_by_keep

    def keep_scale(self, batch: int, device, dtype=torch.float32) -> Optional[torch.Tensor]:
        if self.drop_prob == 0.0 or not self.training:
            return None
        keep = 1.0 - self.drop_prob
        mask = torch.empty(batch, device=device, dtype=dtype).bernoulli_(keep)
        if keep > 0.0 and self.scale_by_keep:
            mask.div_(keep)
        return mask

    def forward(self, x):
        ks = self.keep_scale(x.shape[0], x.device, x.dtype)
        return x if ks is None else x * ks.view((-1,) + (1,) * (x.dim() - 1))


class LayerNorm(nn.Module):
    """cod.py:1025-1049 (channels_last -> F.layer_norm semantics; channels_first -> over dim 1)."""

    def __init__(self, normalized_shape, eps=1e-6, data_format="channels_last"):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(normalized_shape))
        self.bias = nn.Parameter(torch.zeros(normalized_shape))
        self.eps = eps
        self.data_format = data_format
        if self.data_format not in ["channels_last", "channels_first"]:
            raise NotImplementedError
        self.normalized_shape = (normalized_shape,)

    def forward(self, x):
        if _wants_grad(self, x):   # stand-alone differentiable call (weight / bias / input gradients)
            if self.data_format == "channels_first":
                y = TF.LayerNormRowsFn.apply(TF.LayoutFn.apply(x, True), self.weight, self.bias, self.eps)
                return TF.LayoutFn.apply(y, False)
            return TF.LayerNormRowsFn.apply(x, self.weight, self.bias, self.eps)
        return OP.layer_norm(x.contiguous().float(), self.weight.detach(), self.bias.detach(), self.eps,
                             self.data_format == "channels_first")


class ShapePropWeightRegressor(nn.Module):
    """cod.py:1051-1060."""

    def __init__(self, in_channels, latent_dim):
        super(ShapePropWeightRegressor, self).__init__()
        self.latent_dim = latent_dim
        self.reg = nn.Conv2d(in_channels, self.latent_dim * 49, kernel_size=1)

    def forward(self, x):
        return OP.conv1x1_nchw_autograd(x, self.reg.weight, self.reg.bias, True)   # differentiable


class convnext_Block(nn.Module):
    """cod.py:1082-1117."""

    def __init__(self, dim, drop_path=0., layer_scale_init_value=1e-6):
        super().__init__()
        self.dwconv = nn.Conv2d(dim, dim, kernel_size=7, padding=3, groups=dim)
        self.norm = LayerNorm(dim, eps=1e-6)
        self.pwconv1 = nn.Linear(dim, 4 * dim)
        self.act = nn.GELU()
        self.pwconv2 = nn.Linear(4 * dim, dim)
        self.gamma = nn.Parameter(layer_scale_init_value * torch.ones((dim)),
                                  requires_grad=True) if layer_scale_init_value > 0 else None
        self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()

    # x: NHWC fp32 residual stream, updated in place.
    def _forward_nhwc(self, x: torch.Tensor, mode: int) -> torch.Tensor:
        pk = _packed(self)
        B, h, w, C = x.shape
        dw_w = pk.get("dw", [self.dwconv.weight], lambda: self.dwconv.weight.detach().reshape(C, 49).float().contiguous())
        w1 = pk.get(f"w1.{mode}", [self.pwconv1.weight], lambda: _as(self.pwconv1.weight, mode))
        w2 = pk.get(f"w2.{mode}", [self.pwconv2.weight], lambda: _as(self.pwconv2.weight, mode))
        keep = self.drop_path.keep_scale(B, x.device) if isinstance(self.drop_path, DropPath) else None
        gamma = self.gamma.detach() if self.gamma is not None else None
        if mode == BF16 and LN_FOLD and C % 128 == 0 and B * h * w >= 2048:
            # LayerNorm folded into pwconv1: the conv output is stored once (bf16), per-pixel (mean, rstd) come from the
            # stored values, and pwconv1's epilogue applies rstd * (y W'^T - mean * rowsum(W')) + (W1 ln_b + b1)
            dw_wT = pk.get("dwT", [self.dwconv.weight],
                           lambda: self.dwconv.weight.detach().reshape(C, 49).t().float().contiguous())

            def fold():
                w1f = self.pwconv1.weight.detach().float()
                wq = (w1f * self.norm.weight.detach().float()[None, :]).to(torch.bfloat16).contiguous()
                return (wq, wq.float().sum(1).contiguous(),
                        (w1f @ self.norm.bias.detach().float() + self.pwconv1.bias.detach().float()).contiguous())
            wq, col_s, cbias = pk.get("w1.lnfold", [self.pwconv1.weight, self.pwconv1.bias, self.norm.weight, self.norm.bias], fold)
            y, stats = OP.dwconv7_stats_tma(x, dw_wT, self.dwconv.bias.detach(), self.norm.eps)
            if keep is None and C in OP.MLP_FUSED_C and (B * h * w) % 128 == 0:
                # stage 0: both pointwise GEMMs in one kernel, the 4C hidden tensor never reaches HBM
                OP.convnext_mlp_fused_(y.view(-1, C), stats, wq, col_s, cbias, w2, self.pwconv2.bias.detach(), gamma, x)
                return x
            hid = OP.linear_lnfold(y.view(-1, C), wq, cbias, col_s, stats, act=ACT_GELU)
            OP.linear_residual_(hid, w2, self.pwconv2.bias.detach(), gamma, keep, h * w, x)
            return x
        if C % 128 == 0 and B * h * w >= 2048:   # TMA-staged conv + row LayerNorm (large maps)
            dw_wT = pk.get("dwT", [self.dwconv.weight],
                           lambda: self.dwconv.weight.detach().reshape(C, 49).t().float().contiguous())
            ws = _scratch(x.device, x.numel())
            a = OP.dwconv7_ln_tma(x, dw_wT, self.dwconv.bias.detach(), self.norm.weight.detach(),
                                  self.norm.bias.detach(), mode, ws, self.norm.eps)
        else:
            a = OP.dwconv7_ln(x, dw_w, self.dwconv.bias.detach(), self.norm.weight.detach(),
                              self.norm.bias.detach(), mode, self.norm.eps)
        hid = OP.linear(a.view(-1, C), w1, self.pwconv1.bias.detach(), act=ACT_GELU)
        OP.linear_residual_(hid, w2, self.pwconv2.bias.detach(), gamma, keep, h * w, x)
        return x

    def _forward_train(self, x: torch.Tensor, mode: int = F32) -> torch.Tensor:
        """NHWC fp32 in/out with an autograd graph (DropPath mask drawn like timm's, cod.py:1102).
        mode BF16: pointwise GEMMs and their gradients on tcgen05 (bf16 operands, fp32 accumulate)."""
        keep = self.drop_path.keep_scale(x.shape[0], x.device) if isinstance(self.drop_path, DropPath) else None
        M = x.shape[0] * x.shape[1] * x.shape[2]
        fn = TF.ConvNextBlockBf16Fn if (mode == BF16 and TF.tc_rows_ok(M) and x.shape[-1] % 128 == 0) else TF.ConvNextBlockFn
        return fn.apply(x, self.dwconv.weight, self.dwconv.bias, self.norm.weight, self.norm.bias,
                                        self.pwconv1.weight, self.pwconv1.bias, self.pwconv2.weight,
                                        self.pwconv2.bias, self.gamma, keep, self.norm.eps)

    def forward(self, x):
        if _wants_grad(self, x):
            return TF.LayoutFn.apply(self._forward_train(TF.LayoutFn.apply(x, True), _mode(self)), False)
        y = OP.nchw_to_nhwc(x.contiguous().float())
        y = self._forward_nhwc(y, _mode(self))
        return y.permute(0, 3, 1, 2)  # (N,C,H,W) view with channels-last strides


class ShapePropEncoder(nn.Module):
    """cod.py:1119-1177: ConvNeXt-B sized trunk + 4-level fusion head."""

    def __init__(self, in_channels, out_dim):
        super(ShapePropEncoder, self).__init__()
        self.downsample_layers = nn.ModuleList()
        dims = [128, 256, 512, 1024]
        stem = nn.Sequential(
            nn.Conv2d(3, dims[0], kernel_size=4, stride=4),
            LayerNorm(dims[0], eps=1e-6, data_format="channels_first")
        )
        self.downsample_layers.append(stem)
        for i in range(3):
            downsample_layer = nn.Sequential(
                LayerNorm(dims[i], eps=1e-6, data_format="channels_first"),
                nn.Conv2d(dims[i], dims[i + 1], kernel_size=2, stride=2),
            )
            self.downsample_layers.append(downsample_layer)

        self.stages = nn.ModuleList()
        drop_path_rate = 0.4
        depths = [3, 3, 27, 3]
        layer_scale_init_value = 1.0
        dp_rates = [x.item() for x in torch.linspace(0, drop_path_rate, sum(depths))]
        cur = 0
        for i in range(4):
            stage = nn.Sequential(
                *[convnext_Block(dim=dims[i], drop_path=dp_rates[cur + j],
                                 layer_scale_init_value=layer_scale_init_value) for j in range(depths[i])]
            )
            self.stages.append(stage)
            cur += depths[i]

        self.convs = nn.ModuleList()
        for i in range(4):
            self.convs.append(nn.Conv2d(dims[i], out_dim, 1))
        self.fusion_conv = nn.Conv2d(out_dim * 4, out_dim, 1)
        self.dims = dims
        self.out_dim = out_dim

    def _pyramid(self, image: torch.Tensor, grid: Optional[torch.Tensor], mode: int) -> List[torch.Tensor]:
        """Stem + stages on NHWC fp32; returns the four stage outputs (cod.py:1165-1169)."""
        pk = _packed(self)
        st_conv, st_ln = self.downsample_layers[0][0], self.downsample_layers[0][1]
        w0 = pk.get("stem", [st_conv.weight], lambda: st_conv.weight.detach().reshape(self.dims[0], 48).float().contiguous())
        if mode == BF16 and self.dims[0] % 128 == 0 and image.shape[-1] % 4 == 0:
            # tcgen05 stem: bf16 patches (K = 48) x weights -> fp32, LayerNorm rows in place
            w0b = pk.get("stem.bf16", [st_conv.weight], lambda: w0.to(torch.bfloat16))
            B, _, H, W = image.shape
            patches = OP.stem_patches(image, grid, BF16)
            if self.dims[0] == 128 and patches.shape[0] >= 256:
                # the row LayerNorm in the GEMM's epilogue: the fp32 map is written once instead of written, read and rewritten
                x = OP.linear_ln(patches, w0b, st_conv.bias.detach().float(), st_ln.weight.detach().float(),
                                 st_ln.bias.detach().float(), st_ln.eps).view(B, H // 4, W // 4, self.dims[0])
            else:
                x = OP.linear(patches, w0b, st_conv.bias.detach(), out_dtype=F32)
                x = OP.ln_rows_(x, st_ln.weight.detach(), st_ln.bias.detach(), st_ln.eps).view(B, H // 4, W // 4, self.dims[0])
        else:
            x = OP.stem(image, grid, w0, st_conv.bias.detach(), st_ln.weight.detach(), st_ln.bias.detach(), st_ln.eps)
        outs = []
        for i in range(4):
            if i > 0:
                ln, conv = self.downsample_layers[i][0], self.downsample_layers[i][1]
                B, h, w, C = x.shape
                wd = pk.get(f"ds{i}.{mode}", [conv.weight],
                            lambda conv=conv, C=C: _as(conv.weight.detach().permute(0, 2, 3, 1).reshape(2 * C, 4 * C), mode))
                a = OP.ln_patchify(x, ln.weight.detach(), ln.bias.detach(), mode, ln.eps)
                x = OP.linear(a, wd, conv.bias.detach(), out_dtype=F32).view(B, h // 2, w // 2, 2 * C)
            for blk in self.stages[i]:
                x = blk._forward_nhwc(x, mode)
            outs.append(x)
        return outs

    def _head(self, outs: List[torch.Tensor], want_nchw: bool, pad_to: int = 0, mode: int = F32):
        """cod.py:1171-1176 -> embedding3 as (nhwc fp32, nchw fp32 | None, padded bf16 | None)."""
        pk = _packed(self)
        B = outs[0].shape[0]
        levels, hw = [], []
        L = self.out_dim
        fw = self.fusion_conv.weight
        for i, o in enumerate(outs):
            conv = self.convs[i]
            # fusion conv folded into the head projection (both 1x1, and a 1x1 conv commutes with the bilinear
            # up-sample): z_i = x_i (Wf_i Wh_i)^T + Wf_i bh_i, so the 96 -> 24 product at full resolution is gone
            wl = pk.get(f"headf{i}", [conv.weight, fw],
                        lambda conv=conv, i=i: (fw.detach().reshape(L, 4 * L)[:, i * L:(i + 1) * L].float()
                                                @ conv.weight.detach().reshape(L, -1).float()).contiguous())
            bl = pk.get(f"headfb{i}", [conv.bias, fw],
                        lambda conv=conv, i=i: (fw.detach().reshape(L, 4 * L)[:, i * L:(i + 1) * L].float()
                                                @ conv.bias.detach().float()).contiguous())
            a = o.view(-1, o.shape[-1])
            if mode == BF16 and L % 8 == 0 and L <= 64:
                # tcgen05 projection (N = 24) straight from the fp32 stage output: TF32 products, no bf16 copy
                levels.append(OP.linear_tf32(a, wl, bl))
            else:
                levels.append(OP.linear(a, wl, bl, out_dtype=F32))
            hw.append((o.shape[1], o.shape[2]))
        return OP.fusion_sum(levels, hw, self.fusion_conv.bias.detach(), B, want_nhwc=True, want_nchw=want_nchw,
                             pad_to=pad_to)

    def _forward_train(self, image: torch.Tensor, grid: Optional[torch.Tensor], mode: int = F32) -> torch.Tensor:
        """Autograd-building path: returns embedding3 as NHWC (B,h0,w0,out_dim).  mode F32 = exact
        CUDA-core path; BF16 = trunk GEMMs (forward, dgrad, wgrad) on tcgen05."""
        st_conv, st_ln = self.downsample_layers[0][0], self.downsample_layers[0][1]
        x = TF.StemFn.apply(image, grid, st_conv.weight, st_conv.bias, st_ln.weight, st_ln.bias, st_ln.eps)
        levels = []
        for i in range(4):
            if i > 0:
                ln, conv = self.downsample_layers[i][0], self.downsample_layers[i][1]
                Mo = x.shape[0] * (x.shape[1] // 2) * (x.shape[2] // 2)
                ds = TF.DownsampleBf16Fn if (mode == BF16 and TF.tc_rows_ok(Mo)) else TF.DownsampleFn
                x = ds.apply(x, ln.weight, ln.bias, conv.weight, conv.bias, ln.eps)
            for blk in self.stages[i]:
                x = blk._forward_train(x, mode)
            levels.append(TF.LinearFn.apply(x, self.convs[i].weight, self.convs[i].bias))
        return TF.FusionFn.apply(levels[0], levels[1], levels[2], levels[3], self.fusion_conv.weight,
                                 self.fusion_conv.bias)

    def forward(self, x):
        if _wants_grad(self, x):
            return TF.LayoutFn.apply(self._forward_train(x, None, _mode(self)), False)
        outs = self._pyramid(x.contiguous().float(), None, _mode(self))
        _, nchw, _ = self._head(outs, want_nchw=True, mode=_mode(self))
        return nchw


class MessagePassing(nn.Module):
    """cod.py:1180-1208.  ``img_size`` keeps the reference attribute; the fused encoder path
    up-samples to the actual image size instead of the hard-coded 384."""

    def __init__(self, latent_dim, img_size=384, k=7, max_step=4, sym_norm=False):
        super(MessagePassing, self).__init__()
        if k != 7:
            raise NotImplementedError("MessagePassing kernels are built for k=7 (cod.py:1181)")
        if sym_norm:
            raise NotImplementedError("sym_norm branch is dead code in the reference (cod.py:1194-1198)")
        self.k = k
        self.size = k * k
        self.max_step = max_step
        self.sym_norm = sym_norm
        self.img_size = img_size
        self.conv = nn.Conv2d(latent_dim, 3, 1)

    def forward(self, input, weight):
        n, c, h, w = input.size()
        steps = max(h, w) if self.max_step < 0 else self.max_step
        # every step is an autograd.Function backed by the CUDA kernels: differentiable w.r.t.
        # input, weight and self.conv (backward obligations of row a6, SURVEY.md 8a)
        x = OP.message_passing_core(input, weight, steps, 1e-5)
        x = OP.conv1x1_nchw_autograd(x, self.conv.weight, self.conv.bias, False)
        size = self.img_size if isinstance(self.img_size, (tuple, list)) else (self.img_size, self.img_size)
        return OP.resize_bilinear_nchw_autograd(x, size)


_pack_conv3 = DB.pack_conv3
_fold_conv3_bilinear = DB.fold_conv3_bilinear
_pad_taps_bf16 = DB.pad_taps_bf16
_pad_rows = DB.pad_rows
_fold_params = DB.fold_params


class ShapePropDecoder(nn.Module):
    """cod.py:1210-1226."""

    def __init__(self, out_dim, latent_dim):
        super(ShapePropDecoder, self).__init__()
        dilation = 1
        self.decoder = nn.Sequential(
            nn.Conv2d(latent_dim, latent_dim, kernel_size=3, stride=1, padding=dilation, dilation=dilation),
            nn.ReLU(True),
            nn.Conv2d(latent_dim, latent_dim, kernel_size=3, stride=1, padding=dilation, dilation=dilation),
            nn.ReLU(True),
            nn.Conv2d(latent_dim, out_dim, kernel_size=3, stride=1, padding=dilation, dilation=dilation),
        )

    def _forward_train(self, emb_nhwc: torch.Tensor) -> torch.Tensor:
        d = self.decoder
        y = TF.Conv3x3Fn.apply(emb_nhwc, d[0].weight, d[0].bias, True)
        y = TF.Conv3x3Fn.apply(y, d[2].weight, d[2].bias, True)
        return TF.Conv3x3Fn.apply(y, d[4].weight, d[4].bias, False)

    def forward(self, embedding):
        if _wants_grad(self, embedding):
            return self._forward_train(TF.LayoutFn.apply(embedding, True)).permute(0, 3, 1, 2)
        return _decode_full([self], OP.nchw_to_nhwc(embedding.contiguous().float()))[0]


def _decoder_front(decoders: Sequence[ShapePropDecoder], emb: torch.Tensor) -> torch.Tensor:
    """conv1+ReLU of all decoders as ONE conv (they share the input), then conv2+ReLU per decoder
    on its 24-channel slice.  emb NHWC (B,h,w,24) fp32 -> (B,h,w,24*D) fp32."""
    B, h, w, L = emb.shape
    D = len(decoders)
    host = decoders[0]
    pk = _packed(host)
    ws = [d.decoder[0].weight for d in decoders]
    key = "c1." + ".".join(str(id(d)) for d in decoders)
    w1 = pk.get(key + ".w", ws, lambda: torch.cat([_pack_conv3(t) for t in ws], 0).contiguous())
    b1 = pk.get(key + ".b", [d.decoder[0].bias for d in decoders],
                lambda: torch.cat([d.decoder[0].bias.detach().float() for d in decoders]).contiguous())
    h1 = OP.conv_nhwc(emb, w1, b1, L, (h, w), 3, 1, -1, act=ACT_RELU)
    h2 = torch.empty_like(h1)
    for i, d in enumerate(decoders):
        w2 = _packed(d).get("c2", [d.decoder[2].weight], lambda d=d: _pack_conv3(d.decoder[2].weight))
        OP.conv_nhwc(h1[..., i * L:(i + 1) * L], w2, d.decoder[2].bias.detach(), L, (h, w), 3, 1, -1,
                     act=ACT_RELU, out=h2[..., i * L:(i + 1) * L], Cout=L)
    return h2


def _decoder_front_bf16(decoders: Sequence[ShapePropDecoder], emb_pad: torch.Tensor) -> torch.Tensor:
    """tcgen05 path: emb_pad NHWC (B,h,w,32) bf16 (24 latent channels + zero pad) ->
    (D,B,h,w,32) bf16; decoder d owns h2[d], channels [0, 24), the pad channels stay zero."""
    B, h, w, _ = emb_pad.shape
    D = len(decoders)
    L = decoders[0].decoder[0].in_channels
    pk = _packed(decoders[0])
    key = "bf16." + ".".join(str(id(d)) for d in decoders)
    w1 = pk.get(key + ".w1", [d.decoder[0].weight for d in decoders],
                lambda: torch.cat([_pad_taps_bf16(_pack_conv3(d.decoder[0].weight), L, 32) for d in decoders], 0).contiguous())
    b1 = pk.get(key + ".b1", [d.decoder[0].bias for d in decoders],
                lambda: torch.cat([_pad_rows(d.decoder[0].bias, 32) for d in decoders]).contiguous())
    w2 = pk.get(key + ".w2", [d.decoder[2].weight for d in decoders],
                lambda: torch.cat([_pad_taps_bf16(_pack_conv3(d.decoder[2].weight), L, 32) for d in decoders], 0).contiguous())
    b2 = pk.get(key + ".b2", [d.decoder[2].bias for d in decoders],
                lambda: torch.cat([_pad_rows(d.decoder[2].bias, 32) for d in decoders]).contiguous())
    # group-major: every decoder's hidden map is its own dense (B,h,w,32) tensor, so each halo box is made of whole
    # 64-byte pixel rows that no other group's CTA shares (interleaved channel slices read 2.5x their input from DRAM)
    gs = B * h * w * 32
    h1 = torch.empty(D, B, h, w, 32, device=emb_pad.device, dtype=torch.bfloat16)
    OP.conv_nhwc_grouped(emb_pad, w1, b1, 32, (h, w), 3, 1, -1, ACT_RELU, h1, 32 * D, 32, 1, 0, 32 * D, gs)
    h2 = torch.empty_like(h1)
    OP.conv_nhwc_grouped(h1[0], w2, b2, 32, (h, w), 3, 1, -1, ACT_RELU, h2, 32, 32, D, gs, 32, gs)
    return h2


def _decode_tokens_bf16(decoders: Sequence[ShapePropDecoder], h2: torch.Tensor, index0: int,
                        src_hw: Tuple[int, int], grid: Tuple[int, int]) -> List[torch.Tensor]:
    """All decoders of one PVT stage in ONE grouped tcgen05 launch, output (D_s, B, H_s*W_s, E_s) bf16.
    h2: the group-major hidden maps (D_all, B, h, w, 32) of ``_decoder_front_bf16``."""
    B = h2.shape[1]
    D = len(decoders)
    E = decoders[0].decoder[4].out_channels
    L = decoders[0].decoder[4].in_channels
    h, w = src_hw
    fold = _fold_params((h, w), grid)
    pk = _packed(decoders[0])
    key = f"bf16.c3.{grid}." + ".".join(str(id(d)) for d in decoders)
    ws = [d.decoder[4].weight for d in decoders]
    if (h, w) == tuple(grid):
        ks, stride, off = 3, 1, -1
        w3 = pk.get(key, ws, lambda: torch.cat([_pad_taps_bf16(_pack_conv3(t), L) for t in ws], 0).contiguous())
    elif fold is not None:
        ks, stride, off = 4, fold[0], fold[1]
        w3 = pk.get(key, ws, lambda: torch.cat([_pad_taps_bf16(_fold_conv3_bilinear(t), L) for t in ws], 0).contiguous())
    else:
        raise NotImplementedError(f"bf16 prompt injection needs an integer power-of-two ratio, got {(h, w)} -> {grid}")
    b3 = pk.get(key + ".b", [d.decoder[4].bias for d in decoders],
                lambda: torch.cat([d.decoder[4].bias.detach().float() for d in decoders]).contiguous())
    out = torch.empty(D, B, grid[0] * grid[1], E, device=h2.device, dtype=torch.bfloat16)
    OP.conv_nhwc_grouped(h2[index0], w3, b3, 32, grid, ks, stride, off, ACT_NONE, out, E, E, D, h2.stride(0), E,
                         B * grid[0] * grid[1] * E)
    return [out[i] for i in range(D)]


def _decode_full(decoders: Sequence[ShapePropDecoder], emb: torch.Tensor) -> List[torch.Tensor]:
    """Reference-shaped outputs: list of (B,E,h,w) tensors (channels-last strides)."""
    B, h, w, L = emb.shape
    h2 = _decoder_front(decoders, emb)
    outs = []
    for i, d in enumerate(decoders):
        w3 = _packed(d).get("c3", [d.decoder[4].weight], lambda d=d: _pack_conv3(d.decoder[4].weight))
        y = OP.conv_nhwc(h2[..., i * L:(i + 1) * L], w3, d.decoder[4].bias.detach(), L, (h, w), 3, 1, -1)
        outs.append(y.permute(0, 3, 1, 2))
    return outs


def _decode_tokens(decoders: Sequence[ShapePropDecoder], emb: torch.Tensor, grid: Tuple[int, int],
                   h2: Optional[torch.Tensor] = None, index0: int = 0) -> List[torch.Tensor]:
    """Prompts of one PVT stage directly in token layout (B, H_s*W_s, E_s): last conv folded with
    the bilinear down-sample (cod.py:1471) when the ratio allows, else conv + NHWC resize."""
    B, h, w, L = emb.shape
    if h2 is None:
        h2 = _decoder_front(decoders, emb)
        index0 = 0
    outs = []
    fold = _fold_params((h, w), grid)
    for i, d in enumerate(decoders):
        src = h2[..., (index0 + i) * L:(index0 + i + 1) * L]
        conv = d.decoder[4]
        if (h, w) == tuple(grid):
            w3 = _packed(d).get("c3", [conv.weight], lambda conv=conv: _pack_conv3(conv.weight))
            y = OP.conv_nhwc(src, w3, conv.bias.detach(), L, grid, 3, 1, -1)
        elif fold is not None:
            w4 = _packed(d).get("c3fold", [conv.weight], lambda conv=conv: _fold_conv3_bilinear(conv.weight))
            y = OP.conv_nhwc(src, w4, conv.bias.detach(), L, grid, 4, fold[0], fold[1])
        else:
            w3 = _packed(d).get("c3", [conv.weight], lambda conv=conv: _pack_conv3(conv.weight))
            y = OP.resize_nhwc(OP.conv_nhwc(src, w3, conv.bias.detach(), L, (h, w), 3, 1, -1), grid)
        outs.append(y.view(B, grid[0] * grid[1], -1))
    return outs


class prompt_encoder(nn.Module):
    """cod.py:1228-1306."""

    def __init__(self, latent_dim, embed_dim, depth, fusion=False):
        super(prompt_encoder, self).__init__()
        self.embed_dim = embed_dim
        self.depth = depth
        self.propagation_weight_regressor = ShapePropWeightRegressor(3, latent_dim)
        self.encoder1 = nn.Conv2d(1, latent_dim, 1)
        self.encoder2 = ShapePropEncoder(3, 24)
        self.adaptor = nn.Conv2d(6, 3, 1)   # unused by forward, kept for the checkpoint layout (cod.py:1251)
        self.message_passing = MessagePassing(latent_dim, img_size=384, sym_norm=False)
        self.freq_nums = 0.3
        self.latent_dim = latent_dim

    def fft(self, x, rate):
        """cod.py:1256-1271."""
        return OP.fft_highpass(x.contiguous().float(), rate)

    def _forward_fused(self, image: torch.Tensor, cues: torch.Tensor, mode: int, want_nchw: bool = True,
                       pad_to: int = 0):
        H = 12                                                                    # cod.py:1283
        image = image.contiguous().float()
        cues = cues.contiguous().float()
        # :1288; bf16 mode: the projector products on tcgen05 (two-term bf16 split, fp32-accurate)
        x = OP.fft_highpass(image, self.freq_nums, tensor_cores=(mode == BF16))
        reg = self.propagation_weight_regressor.reg
        mp = self.message_passing
        pk = _packed(self)
        reg_w = pk.get("reg", [reg.weight], lambda: reg.weight.detach().reshape(reg.out_channels, 3).float().contiguous())
        enc_w = pk.get("enc1", [self.encoder1.weight], lambda: self.encoder1.weight.detach().reshape(-1).float().contiguous())
        mp_w = pk.get("mpc", [mp.conv.weight], lambda: mp.conv.weight.detach().reshape(3, -1).float().contiguous())
        steps = H if mp.max_step < 0 else mp.max_step
        grid3, _, _ = OP.diffusion_front(x, cues, reg_w, reg.bias.detach(), enc_w, self.encoder1.bias.detach(),
                                         mp_w, mp.conv.bias.detach(), grid=H, steps=steps)   # :1295-1298
        outs = self.encoder2._pyramid(image, grid3, mode)                         # :1302 (+image fused in the stem)
        nhwc, nchw, pad = self.encoder2._head(outs, want_nchw=want_nchw, pad_to=pad_to, mode=mode)
        return x, nhwc, nchw, pad

    def _forward_train(self, image: torch.Tensor, cues: torch.Tensor, mode: Optional[int] = None):
        """Training path (cod.py:1288-1302 op by op, each an autograd Function on the CUDA kernels):
        returns (embedding1, embedding3 NHWC)."""
        mode = _mode(self) if mode is None else mode
        H = 12
        image = image.contiguous().float()
        x = self.fft(image, self.freq_nums)                                            # no parameter upstream
        xx = OP.resize_nchw(x, (H, H), bilinear=False)                                 # nearest, :1295
        weights = self.propagation_weight_regressor(xx)                                # :1296
        # :1297-1298 with the two linear maps swapped (1x1 conv and bilinear resize commute, SURVEY.md
        # appendix A): the 24-channel full-resolution tensor and its gradient are never materialised
        c12 = OP.resize_bilinear_nchw_autograd(cues.contiguous().float(), (H, H))
        d12 = OP.conv1x1_nchw_autograd(c12, self.encoder1.weight, self.encoder1.bias, False)
        mp = self.message_passing
        steps = H if mp.max_step < 0 else mp.max_step
        core = OP.message_passing_core(d12, weights, steps, 1e-5)
        grid3 = OP.conv1x1_nchw_autograd(core, mp.conv.weight, mp.conv.bias, False)     # :1206 (up-sample fused in the stem)
        return x, self.encoder2._forward_train(image, grid3, mode)                     # :1302

    def forward(self, image, cues, cross=False):
        if _wants_grad(self, cues):
            x, emb3 = self._forward_train(image, cues)
            return x, TF.LayoutFn.apply(emb3, False)
        x, _, emb3, _ = self._forward_fused(image, cues, _mode(self), want_nchw=True)
        return x, emb3


class prompt_decoder(nn.Module):
    """cod.py:1308-1323."""

    def __init__(self, latent_dim, embed_dim, depth, fusion=False):
        super(prompt_decoder, self).__init__()
        self.depth = depth
        self.decoder = nn.Sequential(*[ShapePropDecoder(embed_dim, 24) for i in range(depth)])

    def forward(self, embedding, cross=False):
        if _wants_grad(self, embedding):
            emb = TF.LayoutFn.apply(embedding, True)
            return [d._forward_train(emb).permute(0, 3, 1, 2) for d in self.decoder]
        emb = OP.nchw_to_nhwc(embedding.contiguous().float())
        return _decode_full(list(self.decoder), emb)


# ------------------------------------------------------------------------------------------------
def init_weights_(module: nn.Module) -> None:
    """``PyramidVisionTransformerImpr._init_weights`` (cod.py:1401-1414), applied per sub-module."""
    if isinstance(module, nn.Linear):
        nn.init.trunc_normal_(module.weight, std=.02)
        if module.bias is not None:
            nn.init.constant_(module.bias, 0)
    elif isinstance(module, nn.LayerNorm):
        nn.init.constant_(module.bias, 0)
        nn.init.constant_(module.weight, 1.0)
    elif isinstance(module, nn.Conv2d):
        fan_out = module.kernel_size[0] * module.kernel_size[1] * module.out_channels
        fan_out //= module.groups
        module.weight.data.normal_(0, math.sqrt(2.0 / fan_out))
        if module.bias is not None:
            module.bias.data.zero_()


def build_texture_diffuser(seed: Optional[int] = None, embed_dims=PVT_EMBED_DIMS, depths=PVT_DEPTHS,
                           latent_dim: int = 24):
    """The two members ``PyramidVisionTransformerImpr.__init__`` creates for the texture diffuser
    (cod.py:1394-1396), initialised the way ``self.apply(self._init_weights)`` does (:1399)."""
    if seed is not None:
        torch.manual_seed(seed)
    enc = prompt_encoder(latent_dim, list(embed_dims), list(depths), True)
    dec = nn.Sequential(*[prompt_decoder(latent_dim, embed_dims[i], depths[i], True) for i in range(len(depths))])
    enc.apply(init_weights_)
    dec.apply(init_weights_)
    return enc, dec


def pvt_token_grids(img_hw: Sequence[int]) -> List[Tuple[int, int]]:
    """Token grids of the four PVT-v2 stages (OverlapPatchEmbed 7/4/3 then 3/2/1 x3, cod.py:1350-1357)."""
    h, w = int(img_hw[0]), int(img_hw[1])
    h, w = (h + 6 - 7) // 4 + 1, (w + 6 - 7) // 4 + 1
    out = [(h, w)]
    for _ in range(3):
        h, w = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
        out.append((h, w))
    return out


def texture_prompts_train(enc: "prompt_encoder", dec: nn.Sequential, image: torch.Tensor, depth: torch.Tensor,
                          precision: Optional[str] = None):
    """Same contract as `texture_prompts`, building an autograd graph.  precision "fp32" = exact path,
    "bf16" = trunk GEMMs on tcgen05 (None: follow set_precision / torch.autocast)."""
    mode = _mode(enc) if precision is None else (BF16 if precision == "bf16" else F32)
    emb1, emb3 = enc._forward_train(image, depth, mode)            # emb3: NHWC
    grids = pvt_token_grids(image.shape[-2:])
    B = image.shape[0]
    if DB.bank_supported(tuple(emb3.shape[1:3]), grids):
        # all 16 decoders + the folded injection as one Function (tokens bf16 in bf16 mode)
        cfg = {"stages": [(len(dec[s].decoder), tuple(grids[s])) for s in range(len(dec))], "mode": mode}
        params = [t for s in range(len(dec)) for d in dec[s].decoder
                  for t in (d.decoder[0].weight, d.decoder[0].bias, d.decoder[2].weight, d.decoder[2].bias,
                            d.decoder[4].weight, d.decoder[4].bias)]
        flat = DB.DecoderBankFn.apply(emb3, cfg, *params)
        tokens, i = [], 0
        for s in range(len(dec)):
            n = len(dec[s].decoder)
            tokens.append(list(flat[i:i + n]))
            i += n
        return emb1, TF.LayoutFn.apply(emb3, False), tokens
    tokens = []
    for s in range(len(dec)):
        row = []
        for d in dec[s].decoder:
            y = d._forward_train(emb3)                             # (B,h,w,E)
            if tuple(y.shape[1:3]) != tuple(grids[s]):
                y = TF.ResizeNHWCFn.apply(y, grids[s])
            row.append(y.reshape(B, grids[s][0] * grids[s][1], -1))
        tokens.append(row)
    return emb1, TF.LayoutFn.apply(emb3, False), tokens


@torch.no_grad()
def texture_prompts(enc: "prompt_encoder", dec: nn.Sequential, image: torch.Tensor, depth: torch.Tensor,
                    precision: Optional[str] = None, want_embedding3: bool = True):
    """Inference entry (fused kernels, no autograd graph).  Training uses `texture_prompts_train`
    or the module forwards, which switch to the autograd Functions when a graph is requested."""
    return _texture_prompts_infer(enc, dec, image, depth, precision, want_embedding3)


def _texture_prompts_infer(enc: "prompt_encoder", dec: nn.Sequential, image: torch.Tensor, depth: torch.Tensor,
                           precision: Optional[str] = None, want_embedding3: bool = True):
    """The hot path as ``forward_features`` drives it (cod.py:1467-1505) minus the PVT blocks:
    returns ``(embedding1, embedding3, tokens)`` with ``tokens[s][i]`` the (B, H_s*W_s, E_s)
    tensor the reference adds to the stage-s token stream before block i
    (``x = blk(x + prompt[i], H, W)``)."""
    mode = _mode(enc) if precision is None else (BF16 if precision == "bf16" else F32)
    grids = pvt_token_grids(image.shape[-2:])
    all_dec = [d for s in range(len(dec)) for d in dec[s].decoder]
    src_hw = (image.shape[-2] // 4, image.shape[-1] // 4)
    tc_ok = mode == BF16 and all(tuple(g) == src_hw or _fold_params(src_hw, g) is not None for g in grids)
    emb1, nhwc, nchw, pad = enc._forward_fused(image, depth, mode, want_nchw=want_embedding3,
                                               pad_to=32 if tc_ok else 0)
    tokens, idx = [], 0
    if tc_ok:     # decoders on tcgen05 (bf16 operands, fp32 accumulate), 6 launches for all 16 decoders
        h2 = _decoder_front_bf16(all_dec, pad)
        for s in range(len(dec)):
            ds = list(dec[s].decoder)
            tokens.append(_decode_tokens_bf16(ds, h2, idx, src_hw, grids[s]))
            idx += len(ds)
        return emb1, nchw, tokens
    h2 = _decoder_front(all_dec, nhwc)
    for s in range(len(dec)):
        ds = list(dec[s].decoder)
        tokens.append(_decode_tokens(ds, nhwc, grids[s], h2=h2, index0=idx))
        idx += len(ds)
    return emb1, nchw, tokens
