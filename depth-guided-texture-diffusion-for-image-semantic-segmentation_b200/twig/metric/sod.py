"""MAE, S-measure, F-measure and E-measure (twig/metric/{MAE,Smeasure,Fmeasure,Emeasure}.py:18-36: the four
evaluators of config/cod.yml:123-128) and the weighted F-measure of Margolin et al. (CVPR 2014) computed by
csrc/metric_ops.cu.

The reference moves prediction and label to the host and loops over images in numpy (pysodmetrics 1.3.1); here
a batch is four kernel launches on the tensors `cod.forward(mode='predict')` returns, and 16 bytes per image come
back.  The wrappers keep the reference's protocol, including its quirk that every batch records the evaluator's
RUNNING mean over all images seen so far and `compute_metrics` averages those records (Smeasure.py:30-36).
mmengine's `BaseMetric` (collection across ranks) is runner plumbing and out of scope (SURVEY 8).

`sod_metrics_full` and `SODEvaluator` give the whole table that COD papers report (pysodmetrics' `get_results()`:
adaptive, mean and max F- and E-measure, precision and recall curves, next to S, MAE and F^w) from one pass per batch,
without a host synchronisation.

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

__all__ = ["sod_metrics", "sod_metrics_full", "weighted_fmeasure", "MAE", "Smeasure", "Fmeasure", "Emeasure",
           "WeightedFmeasure", "SODEvaluator"]

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


def sod_metrics_full(pred: Maps, gt: Maps) -> Tuple[torch.Tensor, torch.Tensor]:
    """pred, gt as for `sod_metrics` -> (vals, curves) float64: vals (B, 4) = per-image MAE, S-measure, adaptive
    F-measure and adaptive E-measure (pysodmetrics `cal_adaptive_fm` / `cal_adaptive_em`: the prediction binarised at
    min(2 * mean, 1)); curves (B, 4, 256) = changeable F-measure, E-measure, precision and recall (entry i = threshold
    255 - i).  MAE, S and the F / E curves are bit-identical to `sod_metrics(pred, gt, curves=True)`."""
    pred, gt, sizes = _batch(pred, gt)
    B, _, H, W = pred.shape
    ws = torch.empty(int(capi.load().dgtd_sod_metrics_full_ws_bytes(B, H, W)), device=pred.device, dtype=torch.uint8)
    vals = torch.empty(B, 4, device=pred.device, dtype=torch.float64)
    cur = torch.empty(B, 4, 256, device=pred.device, dtype=torch.float64)
    if sizes is None:
        call("dgtd_sod_metrics_full_fwd", ptr(pred), ptr(gt), ptr(ws), ptr(vals), ptr(cur), B, H, W, stream())
    else:
        call("dgtd_sod_metrics_full_sized_fwd", ptr(pred), ptr(gt), ptr(sizes), ptr(ws), ptr(vals), ptr(cur), B, H, W,
             stream())
    return vals, cur


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


class SODEvaluator:
    """The whole COD table in one evaluator: per batch one `sod_metrics_full` and one `weighted_fmeasure` call, with
    the sums kept on the device (no host synchronisation until `evaluate`).

    It aggregates like pysodmetrics' `get_results()`: per-image values (S, F^w, MAE, adaptive E and F) are averaged
    over every image seen, and the F / E / precision / recall curves are averaged over images before the max or the
    mean over thresholds is taken.  It does NOT follow the reference wrappers' protocol (MAE, Smeasure, Fmeasure,
    Emeasure above), which record a running mean per batch and average those records: with batches of unequal
    weight that protocol gives other numbers.  `evaluate()` returns Smeasure, wFmeasure, MAE, adpEm, meanEm, maxEm,
    adpFm, meanFm and maxFm as floats, and the mean curves `fm_curve`, `em_curve`, `precision` and `recall` as
    (256,) float64 numpy arrays (entry i = threshold 255 - i), e.g. for PR plots."""
    default_prefix = 'COD'

    def __init__(self, collect_device: str = 'cpu', prefix: Optional[str] = None, data_range: Optional[float] = 1.0):
        self.collect_device = collect_device
        self.prefix = prefix or self.default_prefix
        self._vals: Optional[torch.Tensor] = None      # sums over images: MAE, S, adaptive F, adaptive E, F^w
        self._curves: Optional[torch.Tensor] = None    # sums over images of the four curves
        self._count = 0

    def process(self, data_batch, data_samples: Tuple[Maps, Maps]) -> None:
        # a list is packed once and its sizes uploaded once for both calls
        pred, gt = (x if isinstance(x, PaddedBatch) else _detached(x) if isinstance(x, torch.Tensor)
                    else PaddedBatch.from_list(x) for x in data_samples)
        vals, cur = sod_metrics_full(pred, gt)
        wfm = weighted_fmeasure(pred, gt)
        v = torch.cat([vals.sum(0), wfm.sum(0, keepdim=True)])
        c = cur.sum(0)
        self._vals = v if self._vals is None else self._vals + v
        self._curves = c if self._curves is None else self._curves + c
        self._count += vals.shape[0]

    def evaluate(self) -> dict:
        if self._count == 0:
            raise ValueError("SODEvaluator.evaluate: no image has been processed")
        v = (self._vals / self._count).cpu().numpy()
        fm, em, p, r = (self._curves / self._count).cpu().numpy()
        return {"Smeasure": float(v[1]), "wFmeasure": float(v[4]), "MAE": float(v[0]),
                "adpEm": float(v[3]), "meanEm": float(em.mean()), "maxEm": float(em.max()),
                "adpFm": float(v[2]), "meanFm": float(fm.mean()), "maxFm": float(fm.max()),
                "fm_curve": fm, "em_curve": em, "precision": p, "recall": r}
