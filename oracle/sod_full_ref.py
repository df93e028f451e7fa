"""CPU restatement of the rest of the COD table of pysodmetrics 1.3.1: the adaptive F-measure and E-measure
(`Fmeasure.cal_adaptive_fm`, `Emeasure.cal_adaptive_em`), the precision and recall curves (`Fmeasure.cal_pr`) and the
aggregate of `get_results()` (adp, mean and max F and E, precision and recall curves), next to S, MAE and F^w.

TEST INFRASTRUCTURE ONLY: imported by tests/ and tools/; never by the product path.

**Parity unpinned** against the library itself, as for oracle/metrics_ref.py: pysodmetrics is not installed here.
tests/test_oracle_sod_full.py pins this module on a literal transcription of the library's formulas and on hand cases.

The adaptive threshold is the library's `min(2 * pred.mean(), 1)` with numpy's own `mean`; `pairwise_sum` restates
the order in which numpy sums it, which the GPU reproduces.  The adaptive counts are taken the way the GPU takes them:
the normalised prediction's re-quantisation to uint8 is strictly increasing on the levels a map can have, so the
pixels at or above the threshold are those whose bin is at least the bin of the lowest level at or above it, one entry
of the flipped cumulative histograms of `cal_pr`.
"""
from __future__ import annotations

from typing import Dict, List, Tuple

import numpy as np

from .metrics_ref import (BETA, EPS, _cum_hists, emeasure_curve_one, fmeasure_curve_one, mae_one, prepare,
                          smeasure_one)
from .wfm_ref import wfm_one


def pairwise_sum(a: np.ndarray) -> float:
    """numpy's `pairwise_sum` (loops_utils.h) of a 1-D float64 array: below 8 elements in order from 0; up to 128,
    eight accumulators r[k] += a[i + k] for i = 8, 16, ... < n - n % 8, combined as ((r0 + r1) + (r2 + r3)) +
    ((r4 + r5) + (r6 + r7)), then the n % 8 rest in order; above 128, split at n / 2 - (n / 2) % 8."""
    x = a.tolist()

    def pw(lo: int, n: int) -> float:
        if n < 8:
            res = 0.0
            for i in range(lo, lo + n):
                res += x[i]
            return res
        if n <= 128:
            r = x[lo:lo + 8]
            i = 8
            while i < n - n % 8:
                for k in range(8):
                    r[k] += x[lo + i + k]
                i += 8
            res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
            for j in range(lo + i, lo + n):
                res += x[j]
            return res
        n2 = n // 2
        n2 -= n2 % 8
        return pw(lo, n2) + pw(lo + n2, n - n2)

    return pw(0, len(x))


def adaptive_threshold(pred: np.ndarray) -> float:
    """`_get_adaptive_threshold(pred, max_value=1)`."""
    return min(2 * pred.mean(), 1)


def _adaptive_counts(pred: np.ndarray, gt: np.ndarray) -> Tuple[int, int]:
    """(foreground, background) pixels of the prediction binarised at the adaptive threshold."""
    above = pred[pred >= adaptive_threshold(pred)]
    if above.size == 0:
        return 0, 0
    fg_w, bg_w = _cum_hists(pred, gt)
    k = 255 - int(above.min() * 255)
    return int(fg_w[k]), int(bg_w[k])


def cal_adaptive_fm(pred: np.ndarray, gt: np.ndarray, beta: float = BETA) -> float:
    """`Fmeasure.cal_adaptive_fm` on prepared maps: 0 when the binary map misses the ground truth."""
    fg, bg = _adaptive_counts(pred, gt)
    if fg == 0:
        return 0.0
    pre = fg / (fg + bg)
    rec = fg / np.count_nonzero(gt)
    return float((1 + beta) * pre * rec / (beta * pre + rec))


def cal_adaptive_em(pred: np.ndarray, gt: np.ndarray) -> float:
    """`Emeasure.cal_adaptive_em` on prepared maps (`cal_em_with_threshold` at the adaptive threshold)."""
    fg_fg, fg_bg = _adaptive_counts(pred, gt)
    size = gt.shape[0] * gt.shape[1]
    gt_fg = np.count_nonzero(gt)
    pred_fg = fg_fg + fg_bg
    pred_bg = size - pred_fg
    if gt_fg == 0:
        total = pred_bg
    elif gt_fg == size:
        total = pred_fg
    else:
        bg_fg = gt_fg - fg_fg
        bg_bg = pred_bg - bg_fg
        mean_pred, mean_gt = pred_fg / size, gt_fg / size
        combos = [(1 - mean_pred, 1 - mean_gt), (1 - mean_pred, 0 - mean_gt),
                  (0 - mean_pred, 1 - mean_gt), (0 - mean_pred, 0 - mean_gt)]
        parts = []
        for numel, (a, b) in zip([fg_fg, fg_bg, bg_fg, bg_bg], combos):
            align = 2 * (a * b) / (a ** 2 + b ** 2 + EPS)
            parts.append((align + 1) ** 2 / 4 * numel)
        total = sum(parts)
    return float(total / (size - 1 + EPS))


def cal_pr(pred: np.ndarray, gt: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """`Fmeasure.cal_pr`: precision and recall at the 256 thresholds (entry i = threshold 255 - i)."""
    tps, bg_w = _cum_hists(pred, gt)
    ps = tps + bg_w
    ps = np.where(ps == 0, 1, ps)
    return tps / ps, tps / max(np.count_nonzero(gt), 1)


def table_one(pred_u8: np.ndarray, gt_u8: np.ndarray) -> Dict[str, object]:
    """Every per-image value of the table for one uint8 (prediction, label) pair."""
    pred, gt = prepare(pred_u8, gt_u8)
    p, r = cal_pr(pred, gt)
    return {"mae": mae_one(pred_u8, gt_u8), "sm": smeasure_one(pred_u8, gt_u8), "wfm": wfm_one(pred_u8, gt_u8),
            "adp_fm": cal_adaptive_fm(pred, gt), "adp_em": cal_adaptive_em(pred, gt),
            "fm": fmeasure_curve_one(pred_u8, gt_u8), "em": emeasure_curve_one(pred_u8, gt_u8), "p": p, "r": r}


class SODTable:
    """pysodmetrics' `MAE`, `Smeasure`, `WeightedFmeasure`, `Fmeasure` and `Emeasure` stepped together:
    `get_results()` averages the per-image values over every image, and the curves over images before the max or
    the mean over thresholds."""

    def __init__(self):
        self.rows: List[Dict[str, object]] = []

    def step(self, pred_u8: np.ndarray, gt_u8: np.ndarray) -> None:
        self.rows.append(table_one(pred_u8, gt_u8))

    def get_results(self) -> Dict[str, object]:
        col = {k: np.array([row[k] for row in self.rows], dtype=np.float64) for k in self.rows[0]}
        fm, em = col["fm"].mean(axis=0), col["em"].mean(axis=0)
        return {"Smeasure": float(col["sm"].mean()), "wFmeasure": float(col["wfm"].mean()),
                "MAE": float(col["mae"].mean()),
                "adpEm": float(col["adp_em"].mean()), "meanEm": float(em.mean()), "maxEm": float(em.max()),
                "adpFm": float(col["adp_fm"].mean()), "meanFm": float(fm.mean()), "maxFm": float(fm.max()),
                "fm_curve": fm, "em_curve": em, "precision": col["p"].mean(axis=0), "recall": col["r"].mean(axis=0)}


def tie_map(h: int, w: int, rng: np.random.Generator) -> Tuple[np.ndarray, int]:
    """A uint8 h x w map with levels 0 and 255 (so normalisation leaves p = u / 255) and a level a such that, in exact
    arithmetic, 2 * mean(u) = a: the adaptive threshold lands on a prediction level and numpy's rounding decides
    whether the pixels at a are foreground.  Returns (map, a); the pixels are in random order."""
    n = h * w
    while True:
        a = int(rng.integers(1, 255))
        cv = int(rng.integers(1, max(2, n // 4)))
        rest = n - 2 - cv
        need = n * a // 2 - 255 - cv * a
        if (n * a) % 2 or rest < 0 or not 0 <= need <= 255 * rest or (rest == 0 and need != 0):
            continue
        vals = rng.integers(0, 256, rest)
        diff = need - int(vals.sum())             # then move random pixels towards 255 (or 0) until the sum is met
        room = (255 - vals) if diff > 0 else vals
        order = rng.permutation(rest)
        moved = np.minimum(room[order], np.maximum(abs(diff) - (np.cumsum(room[order]) - room[order]), 0))
        vals[order] += np.sign(diff) * moved
        u = np.concatenate([[0, 255], np.full(cv, a), vals]).astype(np.uint8)
        assert 2 * int(u.sum(dtype=np.int64)) == n * a
        rng.shuffle(u)
        return u.reshape(h, w), a
