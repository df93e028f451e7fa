"""CPU restatement of the weighted F-measure of pysodmetrics 1.3.1 (`WeightedFmeasure.cal_wfm`, Margolin et al.,
CVPR 2014, beta = 1) and of the exact Euclidean feature transform it needs.

TEST INFRASTRUCTURE ONLY: imported by tests/ and tools/; never by the product path.

Plain numpy, on purpose without SciPy: the library uses `scipy.ndimage.distance_transform_edt` and `convolve`, and
the GPU tests import this module on machines that may not have SciPy.  tests/test_oracle_wfm.py checks it against
SciPy where SciPy is installed.  Quantisation, normalisation and eps follow oracle/metrics_ref.py (`prepare`).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .metrics_ref import EPS, prepare


def nearest_foreground(gt: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Exact Euclidean feature transform of a boolean mask with at least one True pixel: per pixel the squared
    distance to, and the row and column of, the nearest True pixel.  Among equidistant ones the pixel with the
    lowest column, then the lowest row, is taken -- the choice `scipy.ndimage.distance_transform_edt(gt == 0,
    return_indices=True)` makes.  Separable: along each column the nearest foreground row (the lower row on a tie),
    then along each row the column that minimises (x - j)^2 + dy_j^2 (the lower column on a tie)."""
    H, W = gt.shape
    rows = np.arange(H)[:, None]
    big = np.iinfo(np.int64).max // 4
    up = np.maximum.accumulate(np.where(gt, rows, -1), axis=0)
    dn = np.flip(np.minimum.accumulate(np.flip(np.where(gt, rows, big), 0), axis=0), 0)
    near = np.where((up >= 0) & (rows - up <= dn - rows), up, dn)          # == big: no foreground in the column
    dy2 = np.where(near < big, (near - rows) ** 2, big)
    xs = np.arange(W)
    dx2 = (xs[:, None] - xs[None, :]) ** 2                                   # [x, j]
    d2 = np.empty((H, W), np.int64)
    col = np.empty((H, W), np.int64)
    for y in range(H):
        cost = dx2 + dy2[y][None, :]
        j = np.argmin(cost, axis=1)                                          # first minimum: the lower column
        col[y] = j
        d2[y] = cost[xs, j]
    return d2, near[rows, col], col


def _gauss7(sigma: float = 5.0) -> np.ndarray:
    """pysodmetrics `matlab_style_gauss2D((7, 7), sigma=5)`."""
    y, x = np.ogrid[-3.0:4.0, -3.0:4.0]
    h = np.exp(-(x * x + y * y) / (2 * sigma * sigma))
    h[h < np.finfo(h.dtype).eps * h.max()] = 0
    return h / h.sum()


def wfm_one(pred_u8: np.ndarray, gt_u8: np.ndarray, beta: float = 1.0) -> float:
    """pysodmetrics `WeightedFmeasure.cal_wfm` (Margolin et al., CVPR 2014) without SciPy: the feature transform is
    `nearest_foreground` and the 7x7 Gaussian with zero padding is a sum of shifted copies."""
    pred, gt = prepare(pred_u8, gt_u8)
    if not gt.any():
        return 0.0
    d2, r, c = nearest_foreground(gt)
    dst = np.sqrt(d2.astype(np.float64))
    E = np.abs(pred - gt)
    Et = E[r, c]                                   # the foreground pixels are their own nearest foreground
    H, W = gt.shape
    K = _gauss7()
    pad = np.zeros((H + 6, W + 6))
    pad[3:-3, 3:-3] = Et
    EA = np.zeros((H, W))
    for i in range(7):
        for j in range(7):
            EA += K[i, j] * pad[i:i + H, j:j + W]
    min_e_ea = np.where(gt & (EA < E), EA, E)
    bw = np.where(gt, 1.0, 2 - np.exp(np.log(0.5) / 5 * dst))
    ew = min_e_ea * bw
    tpw = np.sum(gt) - np.sum(ew[gt])
    fpw = np.sum(ew[~gt])
    R = 1 - np.mean(ew[gt])
    P = tpw / (tpw + fpw + EPS)
    return float((1 + beta) * R * P / (R + beta * P + EPS))
