"""Hitnet iterative decoder and the `cod` model on top of it (SURVEY.md 8f-2): mirror of cod.py:355-506,
685-807 and cod.py:36-46,118-222.

Same class names, constructor signatures and attribute names as the reference (identical ``state_dict`` keys,
including the never-executed `ca` / `sa` members and the ONE `nn.PReLU()` slope that the default constructor
argument shares between all CABs); every forward runs on libdgtd_ops.so (csrc/hitnet_ops.cu), NHWC fp32 activations.  fp32 mode = exact CUDA-core
implicit GEMMs (the mask-parity path); bf16 mode (`set_precision` / autocast, like the hot path) = tcgen05: the 3x3
convs as implicit GEMMs (one shifted 4-D TMA box per tap, nothing materialised), the 1x1 / 8x8-stride-4 convs
through a bf16 im2col operand; BatchNorm scale folded into the weights, fp32 accumulation and fp32 outputs.
Two paths, like the hot path: with gradients disabled and eval() the fused inference kernels (BatchNorm's running
statistics folded into the conv epilogue, concatenations produced in place); with gradients wanted or in train() the
autograd Functions of ops/functions/hitnet_train_func.py (train-mode BatchNorm with batch statistics and running
updates, every parameter of `cod.forward(mode='loss')` receives its gradient).

The reference's `torch.cat` operands are produced in place: a conv / resize writes straight into its channel
slice of the concatenated tensor (pixel pitch argument of the kernels), nothing is copied twice.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from ..ops.functions import hitnet_func as HF
from ..ops.functions import hitnet_train_func as HT
from ..ops.functions import texture_diffusion_func as OP
from ..ops.capi import BF16
from ..padded import PaddedBatch
from .pvt import pvt_v2_b2
from .texture_diffuser import _mode, _packed, _wants_grad

__all__ = ["BasicConv2d", "ChannelAttention", "SpatialAttention", "CALayer", "CAB", "SAM", "Hitnet", "cod"]


def conv(in_channels, out_channels, kernel_size, bias=False, stride=1):
    """cod.py:401-404."""
    return nn.Conv2d(in_channels, out_channels, kernel_size, padding=(kernel_size // 2), bias=bias, stride=stride)


def _tap_major(w: torch.Tensor) -> torch.Tensor:
    """(O, I, kh, kw) -> (O, kh*kw*I): the K order of the implicit-GEMM loader."""
    return w.detach().float().permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


def _tap_major_padded_bf16(w: torch.Tensor, scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(O, I, 3, 3) -> (O, 9 * Cp) bf16, input channels zero-padded to Cp = roundup(I, 64) (one or two 128-byte
    TMA rows per tap), optional per-output-channel scale (folded BatchNorm)."""
    O, I = w.shape[0], w.shape[1]
    Cp = (I + 63) // 64 * 64
    t = w.detach().float().permute(0, 2, 3, 1)
    if scale is not None:
        t = t * scale[:, None, None, None]
    out = torch.zeros(O, 3, 3, Cp, device=w.device, dtype=torch.float32)
    out[..., :I] = t
    return out.reshape(O, 9 * Cp).to(torch.bfloat16).contiguous()


def _no_training(m: nn.Module) -> None:
    """The fused inference kernels fold BatchNorm's RUNNING statistics; train() goes through `_forward_train`."""
    assert not m.training, f"{type(m).__name__}: the fused inference path was entered in train() mode"


class BasicConv2d(nn.Module):
    """cod.py:355-368: conv (no bias) -> BatchNorm2d (the ReLU member is never applied)."""

    def __init__(self, in_planes, out_planes, kernel_size, stride=1, padding=0, dilation=1):
        super().__init__()
        self.conv = nn.Conv2d(in_planes, out_planes, kernel_size=kernel_size, stride=stride, padding=padding,
                              dilation=dilation, bias=False)
        self.bn = nn.BatchNorm2d(out_planes)
        self.relu = nn.ReLU(inplace=True)

    def _params(self):
        bn = self.bn
        return _packed(self).get("fold", [self.conv.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var],
                                 lambda: self._fold())

    def _fold(self):
        bn = self.bn
        scale = (bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)).contiguous()
        shift = (bn.bias.detach().float() - bn.running_mean.detach().float() * scale).contiguous()
        return _tap_major(self.conv.weight), scale, shift

    def _forward_nhwc(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        _no_training(self.bn)
        assert self.conv.dilation == (1, 1)
        w, scale, shift = self._params()
        k, s, p = self.conv.kernel_size[0], self.conv.stride[0], self.conv.padding[0]
        oh = (x.shape[1] + 2 * p - k) // s + 1
        ow = (x.shape[2] + 2 * p - k) // s + 1
        if _mode(self) == BF16:
            if (k, s, p) == (3, 1, 1):
                wb = _packed(self).get("fold_bf16p", [self.conv.weight, self.bn.weight, self.bn.running_var],
                                       lambda: _tap_major_padded_bf16(self.conv.weight, scale))
                return HF.conv3_tc(x, wb, shift=shift, out=out)
            wb = _packed(self).get("fold_bf16", [self.conv.weight, self.bn.weight, self.bn.running_var],
                                   lambda: (w * scale[:, None]).to(torch.bfloat16).contiguous())
            return HF.conv_affine_tc(x, wb, (oh, ow), k, s, -p, shift=shift, out=out)
        return HF.conv_affine(x, w, (oh, ow), k, s, -p, scale=scale, shift=shift, out=out)

    def _forward_train(self, x: torch.Tensor) -> torch.Tensor:
        """NHWC fp32 in / out under autograd; train(): batch statistics + running update like nn.BatchNorm2d
        (cod.py:362), eval(): the running statistics."""
        assert self.conv.dilation == (1, 1)
        bn = self.bn
        batch_stats = bn.training or bn.running_mean is None
        mom = bn.momentum
        if bn.training and bn.track_running_stats and bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
            if mom is None:
                mom = 1.0 / float(bn.num_batches_tracked)
        update = bn.training and bn.track_running_stats
        k, s, p = self.conv.kernel_size[0], self.conv.stride[0], self.conv.padding[0]
        return HT.ConvBnFn.apply(x, self.conv.weight, bn.weight, bn.bias, bn.running_mean if update or not batch_stats else None,
                                 bn.running_var if update or not batch_stats else None,
                                 (k, s, p, _mode(self), bn.eps, 0.0 if mom is None else mom, batch_stats))

    def forward(self, x):
        if self.bn.training or _wants_grad(self, x):
            from ..ops.functions import train_func as TF
            return TF.LayoutFn.apply(self._forward_train(TF.LayoutFn.apply(x, True)), False)
        return OP.nhwc_to_nchw(self._forward_nhwc(OP.nchw_to_nhwc(x.detach().float().contiguous())))


class ChannelAttention(nn.Module):
    """cod.py:371-386.  Constructed by Hitnet (parameters exist in the checkpoint) but never executed."""

    def __init__(self, in_planes, ratio=16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.max_pool = nn.AdaptiveMaxPool2d(1)
        self.fc1 = nn.Conv2d(in_planes, in_planes // 16, 1, bias=False)
        self.relu1 = nn.ReLU()
        self.fc2 = nn.Conv2d(in_planes // 16, in_planes, 1, bias=False)
        self.sigmoid = nn.Sigmoid()

    def forward(self, x):
        raise NotImplementedError("ChannelAttention is not on the reference's executed path (cod.py:757-758 commented out)")


class SpatialAttention(nn.Module):
    """cod.py:389-404.  Constructed by Hitnet but never executed."""

    def __init__(self, kernel_size=7):
        super().__init__()
        assert kernel_size in (3, 7), 'kernel size must be 3 or 7'
        padding = 3 if kernel_size == 7 else 1
        self.conv1 = nn.Conv2d(2, 1, kernel_size, padding=padding, bias=False)
        self.sigmoid = nn.Sigmoid()

    def forward(self, x):
        raise NotImplementedError("SpatialAttention is not on the reference's executed path (cod.py:757-758 commented out)")


class CALayer(nn.Module):
    """cod.py:413-429."""

    def __init__(self, channel, reduction=16, bias=False):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.conv_du = nn.Sequential(
            nn.Conv2d(channel, channel // reduction, 1, padding=0, bias=bias),
            nn.ReLU(inplace=True),
            nn.Conv2d(channel // reduction, channel, 1, padding=0, bias=bias),
            nn.Sigmoid())

    def _gate(self, x: torch.Tensor) -> torch.Tensor:
        assert self.conv_du[0].bias is None and self.conv_du[2].bias is None, "CALayer(bias=True) is not built"
        w1, w2 = _packed(self).get("w", [self.conv_du[0].weight, self.conv_du[2].weight],
                                   lambda: (self.conv_du[0].weight.detach().float().flatten(1).contiguous(),
                                            self.conv_du[2].weight.detach().float().flatten(1).contiguous()))
        part, hw = HF.channel_sums(x)
        return HF.channel_gate(part, hw, w1, w2)

    def _forward_nhwc(self, x: torch.Tensor) -> torch.Tensor:
        return HF.gated_sum(x, ga=self._gate(x))

    def forward(self, x):
        return OP.nhwc_to_nchw(self._forward_nhwc(OP.nchw_to_nhwc(x.detach().float().contiguous())))


class CAB(nn.Module):
    """cod.py:434-451: conv3 -> act -> conv3 -> CALayer -> + x."""

    def __init__(self, n_feat, kernel_size, reduction, bias, act):
        super().__init__()
        modules_body = [conv(n_feat, n_feat, kernel_size, bias=bias), act, conv(n_feat, n_feat, kernel_size, bias=bias)]
        self.CA = CALayer(n_feat, reduction, bias=bias)
        self.body = nn.Sequential(*modules_body)

    def _forward_nhwc(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        c0, act, c2 = self.body[0], self.body[1], self.body[2]
        assert isinstance(act, nn.PReLU) and act.weight.numel() == 1, "the reference's act is nn.PReLU() (cod.py:686)"
        assert c0.bias is None and c2.bias is None, "CAB(bias=True) is not built"
        w0, w2 = _packed(self).get("w", [c0.weight, c2.weight], lambda: (_tap_major(c0.weight), _tap_major(c2.weight)))
        k = c0.kernel_size[0]
        hw = (x.shape[1], x.shape[2])
        slope = act.weight.detach().float()
        if _mode(self) == BF16 and k == 3:
            b0, b2 = _packed(self).get("w_bf16p", [c0.weight, c2.weight],
                                       lambda: (_tap_major_padded_bf16(c0.weight), _tap_major_padded_bf16(c2.weight)))
            r = HF.conv3_tc(x, b0)
            r = HF.conv3_tc(r, b2, prelu_in=slope)
        elif _mode(self) == BF16:
            b0, b2 = _packed(self).get("w_bf16", [c0.weight, c2.weight],
                                       lambda: (w0.to(torch.bfloat16).contiguous(), w2.to(torch.bfloat16).contiguous()))
            r = HF.conv_affine_tc(x, b0, hw, k, 1, -(k // 2))
            r = HF.conv_affine_tc(r, b2, hw, k, 1, -(k // 2), prelu_in=slope)
        else:
            r = HF.conv_affine(x, w0, hw, k, 1, -(k // 2), prelu=slope)
            r = HF.conv_affine(r, w2, hw, k, 1, -(k // 2))
        return HF.gated_sum(r, ga=self.CA._gate(r), b=x, out=out)

    def _forward_train(self, x: torch.Tensor) -> torch.Tensor:
        c0, act, c2 = self.body[0], self.body[1], self.body[2]
        assert isinstance(act, nn.PReLU) and act.weight.numel() == 1, "the reference's act is nn.PReLU() (cod.py:686)"
        assert c0.bias is None and c2.bias is None and c0.kernel_size == (3, 3), "CAB(bias=True / kernel != 3) is not built"
        du = self.CA.conv_du
        assert du[0].bias is None and du[2].bias is None, "CALayer(bias=True) is not built"
        return HT.CabFn.apply(x, c0.weight, act.weight, c2.weight, du[0].weight, du[2].weight, _mode(self))

    def forward(self, x):
        if _wants_grad(self, x):
            from ..ops.functions import train_func as TF
            return TF.LayoutFn.apply(self._forward_train(TF.LayoutFn.apply(x, True)), False)
        return OP.nhwc_to_nchw(self._forward_nhwc(OP.nchw_to_nhwc(x.detach().float().contiguous())))


class SAM(nn.Module):
    """cod.py:454-506: per input a channel gate `fc(mean)` and a scalar gate `fc_wight(mean)`."""

    def __init__(self, ch_in=32, reduction=16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.fc = nn.Sequential(
            nn.Linear(ch_in, ch_in // reduction, bias=False), nn.ReLU(inplace=True),
            nn.Linear(ch_in // reduction, ch_in, bias=False), nn.Sigmoid())
        self.fc_wight = nn.Sequential(
            nn.Linear(ch_in, ch_in // reduction, bias=False), nn.ReLU(inplace=True),
            nn.Linear(ch_in // reduction, 1, bias=False), nn.Sigmoid())

    def _forward_nhwc(self, x_h: torch.Tensor, x_l: torch.Tensor) -> torch.Tensor:
        ws = [self.fc[0].weight, self.fc[2].weight, self.fc_wight[0].weight, self.fc_wight[2].weight]
        f0, f2, g0, g2 = _packed(self).get("w", ws, lambda: tuple(w.detach().float().contiguous() for w in ws))
        ph, hw_h = HF.channel_sums(x_h)
        pl, hw_l = HF.channel_sums(x_l)
        return HF.gated_sum(x_h, ga=HF.channel_gate(ph, hw_h, f0, f2), sa=HF.channel_gate(ph, hw_h, g0, g2),
                            b=x_l, gb=HF.channel_gate(pl, hw_l, f0, f2), sb=HF.channel_gate(pl, hw_l, g0, g2))

    def _forward_train(self, x_h: torch.Tensor, x_l: torch.Tensor) -> torch.Tensor:
        return HT.SamFn.apply(x_h, x_l, self.fc[0].weight, self.fc[2].weight, self.fc_wight[0].weight,
                              self.fc_wight[2].weight)

    def forward(self, x_h, x_l):
        if _wants_grad(self, x_h, x_l):
            from ..ops.functions import train_func as TF
            return TF.LayoutFn.apply(self._forward_train(TF.LayoutFn.apply(x_h, True), TF.LayoutFn.apply(x_l, True)), False)
        n = lambda t: OP.nchw_to_nhwc(t.detach().float().contiguous())  # noqa: E731
        return OP.nhwc_to_nchw(self._forward_nhwc(n(x_h), n(x_l)))


def _pair(seq: nn.Sequential, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    for i, m in enumerate(seq):
        x = m._forward_nhwc(x, out if i == len(seq) - 1 else None)
    return x


class Hitnet(nn.Module):
    """cod.py:685-807."""

    def __init__(self, channel=32, n_feat=32, scale_unetfeats=32, kernel_size=3, reduction=4, bias=False, act=nn.PReLU()):
        super().__init__()
        self.backbone = pvt_v2_b2()  # [64, 128, 320, 512]
        self.Translayer2_0 = BasicConv2d(64, channel, 1)
        self.Translayer2_1 = BasicConv2d(128, channel, 1)
        self.Translayer3_1 = BasicConv2d(320, channel, 1)
        self.Translayer4_1 = BasicConv2d(512, channel, 1)
        self.ca = ChannelAttention(64)
        self.sa = SpatialAttention()
        self.SAM = SAM()
        self.down05 = nn.Upsample(scale_factor=0.5, mode='bilinear', align_corners=True)
        self.out_SAM = nn.Conv2d(channel, 1, 1)
        self.out_CFM = nn.Conv2d(channel, 1, 1)
        self.decoder_level4 = nn.Sequential(*[CAB(n_feat, kernel_size, reduction, bias=bias, act=act) for _ in range(2)])
        self.decoder_level3 = nn.Sequential(*[CAB(n_feat + scale_unetfeats, kernel_size, reduction, bias=bias, act=act)
                                              for _ in range(2)])
        self.decoder_level2 = nn.Sequential(*[CAB(n_feat + (scale_unetfeats * 2), kernel_size, reduction, bias=bias, act=act)
                                              for _ in range(2)])
        self.upsample = nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True)
        self.downsample_4 = nn.Upsample(scale_factor=0.25, mode='bilinear', align_corners=True)
        self.upsample_4 = nn.Upsample(scale_factor=4, mode='bilinear', align_corners=True)
        self.conv4 = BasicConv2d(3 * channel, channel, 3, padding=1)
        self.decoder_level1 = nn.Sequential(*[CAB(64, kernel_size, reduction, bias=bias, act=act) for _ in range(2)])
        self.compress_out = BasicConv2d(2 * channel, channel, kernel_size=8, stride=4, padding=2)
        self.compress_out2 = BasicConv2d(2 * channel, channel, kernel_size=1)
        self.channel = channel

    # ------------------------------------------------------------------------------------------------
    def _head(self, m: nn.Conv2d):
        return _packed(m).get("w", [m.weight, m.bias], lambda: (m.weight.detach().float().reshape(-1).contiguous(),
                                                                 m.bias.detach().float().contiguous()))

    @torch.no_grad()
    def decode(self, feats: Sequence[torch.Tensor], iterations: int = 4, want_stage_preds: bool = True
               ) -> Tuple[List[torch.Tensor], Optional[torch.Tensor], Tuple[torch.Tensor, torch.Tensor]]:
        """cod.py:752-805 on the four NHWC backbone maps.

        Returns (stage predictions [(B,1,8h,8w)] (empty when not wanted), SAM prediction (B,1,8h,8w) (None when not
        wanted), (out_CFM(cfm_last), out_SAM(sam)) on the stride-8 grid (B,1,h,w): the x8 up-sample of their sum is
        the predict logit map, bilinear interpolation being linear)."""
        assert not self._decoder_training(), "decode() folds the running statistics; train() goes through decode_train()"
        x1, x2, x3, x4 = feats
        B, ch = x1.shape[0], self.channel
        dev = x1.device
        h2, w2 = x2.shape[1], x2.shape[2]
        h3, w3 = x3.shape[1], x3.shape[2]
        h4, w4 = x4.shape[1], x4.shape[2]
        new = lambda h, w, c: torch.empty(B, h, w, c, device=dev, dtype=torch.float32)  # noqa: E731

        cim = _pair(self.decoder_level1, x1)                                   # :760
        cat2 = new(h2, w2, 3 * ch)          # [x2_t | up(x3_feed)]             :791
        cat3 = new(h3, w3, 2 * ch)          # [x3_t | up(x4_feed)]             :785
        fb2 = new(h2, w2, 2 * ch)           # [x2_t | cfm]                     :789
        fb4 = new(4 * h4, 4 * w4, 2 * ch)   # [up4(x4_t) | cfm]                :778
        assert (4 * h4, 4 * w4) == (h2, w2) and (2 * h3, 2 * w3) == (h2, w2), "backbone grids must be 8/16/32 strides"
        self.Translayer2_1._forward_nhwc(x2, out=cat2[..., :ch])               # :763
        self.Translayer3_1._forward_nhwc(x3, out=cat3[..., :ch])               # :764
        x4_t = self.Translayer4_1._forward_nhwc(x4)                            # :765
        cfm_w, cfm_b = self._head(self.out_CFM)
        sam_w, sam_b = self._head(self.out_SAM)

        preds: List[torch.Tensor] = []
        cfm = fb2[..., ch:]
        pr = None
        for it in range(iterations):
            if it > 0:
                HF.resize_ld(x4_t, (4 * h4, 4 * w4), True, out=fb4[..., :ch])   # :778
                HF.copy_channels(cfm, fb4[..., ch:])
                x4_t = self.compress_out._forward_nhwc(fb4)                     # :779
            x4_f = _pair(self.decoder_level4, x4_t)                             # :786
            HF.resize_ld(x4_f, (h3, w3), True, out=cat3[..., ch:])              # :785
            x3_f = _pair(self.decoder_level3, cat3)                             # :786
            if it > 0:
                HF.copy_channels(cat2[..., :ch], fb2[..., :ch])
                self.compress_out2._forward_nhwc(fb2, out=cat2[..., :ch])       # :789-790
            HF.resize_ld(x3_f, (h2, w2), True, out=cat2[..., ch:])              # :791
            x2_f = _pair(self.decoder_level2, cat2)                             # :792
            self.conv4._forward_nhwc(x2_f, out=cfm)                             # :793
            if want_stage_preds or it == iterations - 1:
                pr = HF.head1(cfm, cfm_w, cfm_b)                                # :794
                if want_stage_preds:
                    preds.append(OP.resize_nchw(pr, (8 * h2, 8 * w2)))          # :796
        t2 = self.Translayer2_0._forward_nhwc(cim)                              # :800
        t2 = HF.resize_ld(t2, (t2.shape[1] // 2, t2.shape[2] // 2), True)       # :801
        sam = self.SAM._forward_nhwc(cfm, t2)                                   # :802
        p2 = HF.head1(sam, sam_w, sam_b)                                        # :805
        p2_8 = OP.resize_nchw(p2, (8 * h2, 8 * w2)) if want_stage_preds else None   # :806
        return preds, p2_8, (pr, p2)

    def decode_train(self, feats: Sequence[torch.Tensor], iterations: int = 4) -> Tuple[List[torch.Tensor], torch.Tensor]:
        """cod.py:752-806 on the four NHWC backbone maps under autograd (train-mode BatchNorm when the module is in
        train()): ([stage predictions (B,1,8h,8w)], SAM prediction).  The `torch.cat`s are ATen copies here (their
        backward is a slice); everything else runs on libdgtd_ops.so."""
        x1, x2, x3, x4 = feats
        h2, w2 = x2.shape[1], x2.shape[2]
        h3, w3 = x3.shape[1], x3.shape[2]
        h4, w4 = x4.shape[1], x4.shape[2]
        assert (4 * h4, 4 * w4) == (h2, w2) and (2 * h3, 2 * w3) == (h2, w2), "backbone grids must be 8/16/32 strides"
        up = lambda t, hw: HT.ResizeLdFn.apply(t, hw, True)                     # noqa: E731
        pair = lambda seq, t: seq[1]._forward_train(seq[0]._forward_train(t))   # noqa: E731
        cim = pair(self.decoder_level1, x1)                                     # :760
        x2_t = self.Translayer2_1._forward_train(x2)                            # :763
        x3_t = self.Translayer3_1._forward_train(x3)                            # :764
        x4_t = self.Translayer4_1._forward_train(x4)                            # :765
        preds: List[torch.Tensor] = []
        cfm = None
        for it in range(iterations):
            if cfm is not None:
                x4_t = self.compress_out._forward_train(torch.cat((up(x4_t, (4 * h4, 4 * w4)), cfm), -1))   # :778-779
            x4_f = pair(self.decoder_level4, x4_t)                              # :786
            x3_f = pair(self.decoder_level3, torch.cat((x3_t, up(x4_f, (h3, w3))), -1))      # :785-786
            if it > 0:
                x2_t = self.compress_out2._forward_train(torch.cat((x2_t, cfm), -1))         # :789-790
            x2_f = pair(self.decoder_level2, torch.cat((x2_t, up(x3_f, (h2, w2))), -1))      # :791-792
            cfm = self.conv4._forward_train(x2_f)                               # :793
            pr = HT.Head1Fn.apply(cfm, self.out_CFM.weight, self.out_CFM.bias)  # :794
            preds.append(OP.resize_bilinear_nchw_autograd(pr, (8 * h2, 8 * w2)))             # :796
        t2 = self.Translayer2_0._forward_train(cim)                             # :800
        t2 = up(t2, (t2.shape[1] // 2, t2.shape[2] // 2))                       # :801
        sam = self.SAM._forward_train(cfm, t2)                                  # :802
        p2 = HT.Head1Fn.apply(sam, self.out_SAM.weight, self.out_SAM.bias)      # :805
        return preds, OP.resize_bilinear_nchw_autograd(p2, (8 * h2, 8 * w2))    # :806

    def _decoder_training(self) -> bool:
        return any(m.training for m in self.modules() if isinstance(m, nn.BatchNorm2d))

    def forward(self, x, pred_normal):
        """cod.py:743-807 -> (embedding1, [4 stage predictions], prediction2_8).  Builds an autograd graph when
        gradients are wanted; train() uses BatchNorm batch statistics (with or without gradients)."""
        if _wants_grad(self, x):
            emb1, feats = self.backbone._forward_features_train(x, pred_normal)
            preds, p2_8 = self.decode_train(feats)
            return emb1, preds, p2_8
        with torch.no_grad():
            emb1, feats = self.backbone._forward_features_nhwc(x, pred_normal)
            if self._decoder_training():
                preds, p2_8 = self.decode_train(feats)
            else:
                preds, p2_8, _ = self.decode(feats)
            return emb1, preds, p2_8

    @torch.no_grad()
    def predict_logits(self, x, depth, size: Optional[Sequence[int]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """(embedding1, `interpolate(P1[-1] + P2, size)`) of cod.py:148-149 without materialising the unused stage
        predictions: the two 1-channel heads are summed on the stride-8 grid and up-sampled once when `size` is the
        x8 grid (bilinear interpolation is linear)."""
        emb1, feats = self.backbone._forward_features_nhwc(x, depth)
        if self._decoder_training():      # train() under no_grad: batch statistics, like the reference would
            preds, p2_8 = self.decode_train(feats)
            out = _add_planes(preds[-1], p2_8)
            if size is not None and tuple(int(v) for v in size) != tuple(out.shape[-2:]):
                out = OP.resize_nchw(out, (int(size[0]), int(size[1])))
            return emb1, out
        _, p2_8, (pr, p2) = self.decode(feats, want_stage_preds=False)
        H8, W8 = 8 * pr.shape[-2], 8 * pr.shape[-1]
        size = (H8, W8) if size is None else (int(size[0]), int(size[1]))
        out = OP.resize_nchw(_add_planes(pr, p2), (H8, W8))
        if size != (H8, W8):
            out = OP.resize_nchw(out, size)
        return emb1, out


def _add_planes(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a + b for (B,1,H,W) fp32 maps through the gated-sum kernel (planes viewed as NHWC with C = 4)."""
    B, _, H, W = a.shape
    assert (H * W) % 4 == 0
    va, vb = a.view(B, 1, H * W // 4, 4), b.view(B, 1, H * W // 4, 4)
    out = torch.empty_like(a)
    HF.gated_sum(va, b=vb, out=out.view(B, 1, H * W // 4, 4))
    return out


class cod(nn.Module):
    """cod.py:36-222 (the reference derives from mmengine's BaseModel; the runner is out of scope, SURVEY 8).

    `forward(raw, input, label, depth, mode)`: 'predict' -> (sigmoid(output), label) like cod.py:217 without the
    PNG side effects; 'tensor' -> output logits; 'loss' -> {'loss': loss_p1 + loss_P2 + loss_3} of cod.py:135-146
    with an autograd graph to every parameter when gradients are enabled (the training step of cod.py:118-146).

    'predict' with `label` a list of maps of different sizes (the public COD test sets keep each mask at its source
    resolution) predicts the batch once and resizes image b's logits to its own label's size, like cod.py:149 does
    one image at a time.  It returns (probabilities, labels) as two `PaddedBatch` on the input's device, which the
    evaluators of twig/metric take as they are.  'tensor' does not take such labels."""

    def __init__(self, win_size=None, filter_ratio=None, using_depth=None, using_sam=None, finetune=None,
                 binary_thresh=None, pretrain_sam=None, head=None):
        super().__init__()
        self.hitnet = Hitnet()
        self.batch = 0
        self.binary_thresh = binary_thresh

    def forward(self, raw, input, label, depth, mode='loss'):
        if isinstance(input, (tuple, list)):
            input = torch.stack(input, dim=0)
        ragged = (mode in ('predict', 'tensor') and isinstance(label, (tuple, list))
                  and len({tuple(lb.shape[-2:]) for lb in label}) > 1)
        if isinstance(label, (tuple, list)) and not ragged:
            label = torch.stack(label, dim=0)
        if isinstance(depth, (tuple, list)):
            depth = torch.stack(depth, dim=0)
        if ragged:
            if mode == 'tensor':
                raise NotImplementedError("mode='tensor' takes labels of one size only")
            with torch.no_grad():
                labels = PaddedBatch.from_list(label, device=input.device)
                _, output = self.hitnet.predict_logits(input, depth, None)
                return HF.resize_sigmoid_sized(output, labels), labels
        if mode in ('predict', 'tensor'):
            with torch.no_grad():
                size = label.shape[-2:] if label is not None else None
                _, output = self.hitnet.predict_logits(input, depth, size)
                if mode == 'tensor':
                    return output
                return _sigmoid(output), label
        if mode == 'loss':
            from .losses import total_loss
            emb1, P1, P2 = self.hitnet(input, depth)
            return {'loss': total_loss(emb1, P1, P2, input, label.float().contiguous())}
        raise NotImplementedError(f'Unsupported mode {mode}')


def _sigmoid(x: torch.Tensor) -> torch.Tensor:
    return HF.sigmoid(x)
