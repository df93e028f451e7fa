"""MAE, S-measure, F-measure and E-measure (twig/metric/{MAE,Smeasure,Fmeasure,Emeasure}.py:18-36: the four
evaluators of config/cod.yml:123-128) and the weighted F-measure of Margolin et al. (CVPR 2014) computed by
csrc/metric_ops.cu.

The reference moves prediction and label to the host and loops over images in numpy (pysodmetrics 1.3.1); here
a batch is four kernel launches on the tensors `cod.forward(mode='predict')` returns, and 16 bytes per image come
back.  The wrappers keep the reference's protocol, including its quirk that every batch records the evaluator's
RUNNING mean over all images seen so far and `compute_metrics` averages those records (Smeasure.py:30-36).
mmengine's `BaseMetric` (collection across ranks) is runner plumbing and out of scope (SURVEY 8).

Every function and evaluator also takes ground truths of different sizes, as pysodmetrics scores each prediction at
its own ground truth's resolution: a pair of `PaddedBatch` or a pair of lists of per-image maps.  One call then
scores the whole batch, and image b's values are bit-identical to a call on its H_b x W_b maps alone.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple, Union

import torch

from ..ops import capi
from ..ops.capi import call, check_cuda, ptr, stream
from ..padded import PaddedBatch

__all__ = ["sod_metrics", "weighted_fmeasure", "MAE", "Smeasure", "Fmeasure", "Emeasure", "WeightedFmeasure"]

Maps = Union[torch.Tensor, PaddedBatch, Sequence[torch.Tensor]]


def _check_maps(pred: torch.Tensor, gt: torch.Tensor) -> None:
    check_cuda(pred, gt)
    assert pred.dtype == torch.float32 and gt.dtype == torch.float32, "fp32 maps expected (cod.py:217)"
    assert pred.shape == gt.shape and pred.dim() == 4 and pred.shape[1] == 1, (tuple(pred.shape), tuple(gt.shape))


def _batch(pred: Maps, gt: Maps) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
    """-> (pred, gt, sizes): the two (B,1,H,W) buffers and, for maps of different sizes, the device (B, 2) sizes
    (None when every image fills its buffer).  Raises ValueError, before any launch, when pred[b] and gt[b] differ in
    size or a side is below 2."""
    if isinstance(pred, torch.Tensor) and isinstance(gt, torch.Tensor):
        _check_maps(pred, gt)
        return pred, gt, None
    p, g = (x if isinstance(x, PaddedBatch) else PaddedBatch.from_list(x) for x in (pred, gt))
    if p.sizes != g.sizes:
        raise ValueError(f"prediction sizes {p.sizes} differ from ground-truth sizes {g.sizes}")
    if p.data.shape != g.data.shape:
        raise ValueError(f"prediction buffer {tuple(p.data.shape)} differs from ground-truth buffer "
                         f"{tuple(g.data.shape)}")
    _check_maps(p.data, g.data)
    return p.data, g.data, p.device_sizes()


def sod_metrics(pred: Maps, gt: Maps, curves: bool = False):
    """pred, gt (B,1,H,W) fp32 in [0,1] on the GPU -> (B, 2) float64 = per-image (MAE, S-measure); with
    `curves=True` also (B, 2, 256) float64 = per-image changeable F-measure and E-measure curves.  pred and gt may
    also be two `PaddedBatch` or two lists of (1,H,W) / (H,W) maps whose sizes differ from image to image."""
    pred, gt, sizes = _batch(pred, gt)
    B, _, H, W = pred.shape
    ws = torch.empty(int(capi.load().dgtd_sod_metrics_ws_bytes(B, H, W)), device=pred.device, dtype=torch.uint8)
    out = torch.empty(B, 2, device=pred.device, dtype=torch.float64)
    cur = torch.empty(B, 2, 256, device=pred.device, dtype=torch.float64) if curves else None
    if sizes is None:
        call("dgtd_sod_metrics_fwd", ptr(pred), ptr(gt), ptr(ws), ptr(out), ptr(cur), B, H, W, stream())
    else:
        call("dgtd_sod_metrics_sized_fwd", ptr(pred), ptr(gt), ptr(sizes), ptr(ws), ptr(out), ptr(cur), B, H, W,
             stream())
    return (out, cur) if curves else out


def weighted_fmeasure(pred: Maps, gt: Maps) -> torch.Tensor:
    """pred, gt (B,1,H,W) fp32 in [0,1] on the GPU -> (B,) float64 = per-image weighted F-measure (pysodmetrics
    `WeightedFmeasure`, beta = 1; 0 for an empty ground truth).  H and W must both exceed 1.  Takes the same
    per-image-size forms as `sod_metrics`."""
    pred, gt, sizes = _batch(pred, gt)
    B, _, H, W = pred.shape
    ws = torch.empty(int(capi.load().dgtd_sod_wfm_ws_bytes(B, H, W)), device=pred.device, dtype=torch.uint8)
    out = torch.empty(B, device=pred.device, dtype=torch.float64)
    if sizes is None:
        call("dgtd_sod_wfm_fwd", ptr(pred), ptr(gt), ptr(ws), ptr(out), B, H, W, stream())
    else:
        call("dgtd_sod_wfm_sized_fwd", ptr(pred), ptr(gt), ptr(sizes), ptr(ws), ptr(out), B, H, W, stream())
    return out


def _detached(x: Maps) -> Maps:
    return x.detach().float().contiguous() if isinstance(x, torch.Tensor) else x


def _sod_column(column: int):
    return lambda pred, gt: sod_metrics(pred, gt)[:, column]


class _Running:
    """The evaluator keeps every image's value; a batch records the mean over all images seen so far.  `_per_image`
    maps a (pred, gt) batch to its (B,) values."""
    default_prefix = 'COD'
    _per_image = None
    _key = ''
    _name = ''

    def __init__(self, collect_device: str = 'cpu', prefix: Optional[str] = None, data_range: Optional[float] = 1.0):
        self.collect_device = collect_device
        self.prefix = prefix or self.default_prefix
        self.results: List[dict] = []
        self._sum = 0.0
        self._count = 0

    def process(self, data_batch, data_samples: Tuple[torch.Tensor, torch.Tensor]) -> None:
        pred, gt = data_samples
        vals = self._per_image(_detached(pred), _detached(gt))
        for v in vals.cpu().tolist():           # the evaluator's list of per-image values, as a running sum
            self._sum += v
            self._count += 1
        self.results.append({self._key: self._sum / self._count})

    def compute_metrics(self, results: list) -> dict:
        return {self._name: sum(r[self._key] for r in results) / len(results)}

    def evaluate(self) -> dict:
        return self.compute_metrics(self.results)


class _RunningCurve:
    """Fmeasure.py / Emeasure.py: the evaluator keeps every image's 256-threshold curve; a batch records the
    maximum over thresholds of the MEAN curve over all images seen so far."""
    default_prefix = 'COD'
    _row = 0
    _key = ''
    _name = ''

    def __init__(self, collect_device: str = 'cpu', prefix: Optional[str] = None, data_range: Optional[float] = 1.0):
        self.collect_device = collect_device
        self.prefix = prefix or self.default_prefix
        self.results: List[dict] = []
        self._sum: Optional[torch.Tensor] = None      # running sum of curves, kept on the GPU
        self._count = 0

    def process(self, data_batch, data_samples: Tuple[torch.Tensor, torch.Tensor]) -> None:
        pred, gt = data_samples
        _, cur = sod_metrics(_detached(pred), _detached(gt), curves=True)
        batch_sum = cur[:, self._row].sum(0)
        self._sum = batch_sum if self._sum is None else self._sum + batch_sum
        self._count += cur.shape[0]
        self.results.append({self._key: float((self._sum / self._count).max())})

    def compute_metrics(self, results: list) -> dict:
        return {self._name: sum(r[self._key] for r in results) / len(results)}

    def evaluate(self) -> dict:
        return self.compute_metrics(self.results)


class Fmeasure(_RunningCurve):
    """twig/metric/Fmeasure.py."""
    _row, _key, _name = 0, 'fm', 'Fmeasure'


class Emeasure(_RunningCurve):
    """twig/metric/Emeasure.py."""
    _row, _key, _name = 1, 'em', 'Emeasure'


class MAE(_Running):
    """twig/metric/MAE.py."""
    _per_image, _key, _name = staticmethod(_sod_column(0)), 'mae', 'MAE'


class Smeasure(_Running):
    """twig/metric/Smeasure.py."""
    _per_image, _key, _name = staticmethod(_sod_column(1)), 'sm', 'Smeasure'


class WeightedFmeasure(_Running):
    """twig/metric/WeightedFmeasure.py (commented out in the reference): pysodmetrics `WeightedFmeasure`."""
    _per_image, _key, _name = staticmethod(weighted_fmeasure), 'wfm', 'WeightedFmeasure'
