"""The numpy restatement of pysodmetrics' adaptive F- and E-measure and precision / recall curves
(oracle/sod_full_ref.py) against a literal transcription of the library, numpy's summation order of `p.mean()`, and
the re-quantisation argument the adaptive counts rest on."""
import math

import numpy as np
import pytest

from oracle import metrics_ref as M
from oracle import sod_full_ref as F


def _levels_map(rng, shape):
    """A normalised prediction as the library sees it: u8 levels, min-max normalised."""
    u = rng.integers(0, 256, shape).astype(np.uint8)
    return M.prepare(u, np.zeros(shape, np.uint8))[0]


def test_pairwise_sum_is_numpys_mean():
    rng = np.random.default_rng(0)
    shapes = [(1, n) for n in range(1, 140)] + [(2, n // 2) for n in range(4, 300, 2)]
    shapes += [(1, 2 ** k + d) for k in range(3, 21) for d in (-1, 0, 1)]
    shapes += [(37, 53), (61, 2), (2, 1000), (384, 384), (352, 353), (1000, 999), (4000, 3000)]
    for shape in shapes:
        p = _levels_map(rng, shape) if shape[0] * shape[1] > 1 else rng.random(shape)
        assert F.pairwise_sum(p.ravel()) / p.size == p.mean(), shape


def test_requantisation_is_strictly_increasing():
    """For every (min, range) pair a u8 map can have, `(p * 255).astype(np.uint8)` of the normalised levels is strictly
    increasing: a threshold on p is a threshold on the re-quantised bin, so the adaptive counts are one entry of the
    cumulative histograms."""
    u = np.arange(256) / 255.0
    for dmin in range(256):
        for R in range(1, 256 - dmin):
            mn, mx = dmin / 255.0, (dmin + R) / 255.0
            q = ((u[dmin:dmin + R + 1] - mn) / (mx - mn) * 255).astype(np.uint8)
            assert (np.diff(q.astype(np.int64)) > 0).all(), (dmin, R)


def _literal_fm(pred, gt, beta=0.3):
    """pysodmetrics 1.3.1 `Fmeasure.cal_adaptive_fm`, transcribed as published."""
    adaptive_threshold = min(2 * pred.mean(), 1)
    binary_predcition = pred >= adaptive_threshold
    area_intersection = binary_predcition[gt].sum()
    if area_intersection == 0:
        adaptive_fm = 0
    else:
        pre = area_intersection / np.count_nonzero(binary_predcition)
        rec = area_intersection / np.count_nonzero(gt)
        adaptive_fm = (1 + beta) * pre * rec / (beta * pre + rec)
    return adaptive_fm


def _literal_em(pred, gt):
    """pysodmetrics 1.3.1 `Emeasure.cal_adaptive_em` -> `cal_em_with_threshold`, transcribed as published."""
    gt_fg_numel = np.count_nonzero(gt)
    gt_size = gt.shape[0] * gt.shape[1]
    binarized_pred = pred >= min(2 * pred.mean(), 1)
    fg_fg_numel = np.count_nonzero(binarized_pred & gt)
    fg_bg_numel = np.count_nonzero(binarized_pred & ~gt)
    fg___numel = fg_fg_numel + fg_bg_numel
    bg___numel = gt_size - fg___numel
    if gt_fg_numel == 0:
        enhanced_matrix_sum = bg___numel
    elif gt_fg_numel == gt_size:
        enhanced_matrix_sum = fg___numel
    else:
        bg_fg_numel = gt_fg_numel - fg_fg_numel
        bg_bg_numel = bg___numel - bg_fg_numel
        parts_numel = [fg_fg_numel, fg_bg_numel, bg_fg_numel, bg_bg_numel]
        mean_pred_value = fg___numel / gt_size
        mean_gt_value = gt_fg_numel / gt_size
        combinations = [(1 - mean_pred_value, 1 - mean_gt_value), (1 - mean_pred_value, 0 - mean_gt_value),
                        (0 - mean_pred_value, 1 - mean_gt_value), (0 - mean_pred_value, 0 - mean_gt_value)]
        results_parts = []
        for part_numel, combination in zip(parts_numel, combinations):
            align_matrix_value = 2 * (combination[0] * combination[1]) / (combination[0] ** 2 + combination[1] ** 2
                                                                          + M.EPS)
            enhanced_matrix_value = (align_matrix_value + 1) ** 2 / 4
            results_parts.append(enhanced_matrix_value * part_numel)
        enhanced_matrix_sum = sum(results_parts)
    return enhanced_matrix_sum / (gt_size - 1 + M.EPS)


def _hand_cases():
    H, W = 24, 40
    blob = np.zeros((H, W), np.uint8)
    blob[6:18, 10:30] = 255
    rng = np.random.default_rng(7)
    rnd = rng.integers(0, 256, (H, W)).astype(np.uint8)
    full = lambda v: np.full((H, W), v, np.uint8)  # noqa: E731
    return {"empty gt": (rnd, full(0)), "full gt": (rnd, full(255)), "perfect": (blob.copy(), blob),
            "inverted": (255 - blob, blob), "constant 0": (full(0), blob), "constant 51": (full(51), blob),
            "constant 255": (full(255), blob), "constant 0, empty gt": (full(0), full(0))}


def test_adaptive_values_match_the_literal_transcription():
    rng = np.random.default_rng(1)
    cases = list(_hand_cases().values())
    for H, W in ((2, 2), (2, 3), (5, 7), (33, 40), (64, 48), (2, 300), (129, 3)):
        for dens in (0.05, 0.4):
            cases.append((rng.integers(0, 256, (H, W)).astype(np.uint8),
                          (rng.random((H, W)) < dens).astype(np.uint8) * 255))
        lo = int(rng.integers(0, 200))                          # a narrow prediction range
        cases.append((rng.integers(lo, lo + 40, (H, W)).astype(np.uint8),
                      (rng.random((H, W)) < 0.3).astype(np.uint8) * 255))
    for pu, gu in cases:
        pred, gt = M.prepare(pu, gu)
        assert abs(F.cal_adaptive_fm(pred, gt) - _literal_fm(pred, gt)) <= 1e-12, pu.shape
        assert abs(F.cal_adaptive_em(pred, gt) - _literal_em(pred, gt)) <= 1e-12, pu.shape


def test_hand_case_values():
    c = _hand_cases()
    val = {k: (F.cal_adaptive_fm(*M.prepare(*v)), F.cal_adaptive_em(*M.prepare(*v))) for k, v in c.items()}
    assert abs(val["perfect"][0] - 1.0) < 1e-12 and val["inverted"][0] == 0.0
    # constant 0: threshold 0, every pixel is foreground; constant 51 stays un-normalised, 2 * mean is above its only
    # level and no pixel is; constant 255: p = 1 = threshold, every pixel is
    n, fg = 24 * 40, 12 * 20
    assert _literal_fm(*M.prepare(*c["constant 0"])) == val["constant 0"][0]
    assert abs(val["constant 0"][0] - 1.3 * (fg / n) / (0.3 * (fg / n) + 1)) < 1e-12
    assert val["constant 51"][0] == 0.0 and val["constant 255"][0] == val["constant 0"][0]
    assert val["constant 0, empty gt"] == (0.0, 0.0)
    assert abs(val["perfect"][1] - n / (n - 1)) < 1e-12


def test_precision_recall_match_the_published_formulas():
    rng = np.random.default_rng(2)
    for H, W in ((2, 3), (37, 53), (64, 64)):
        pu = rng.integers(0, 256, (H, W)).astype(np.uint8)
        gu = (rng.random((H, W)) < 0.3).astype(np.uint8) * 255
        pred, gt = M.prepare(pu, gu)
        p, r = F.cal_pr(pred, gt)
        q = (pred * 255).astype(np.uint8)
        for i in range(256):                                  # brute force, threshold by threshold
            b = q >= 255 - i
            assert p[i] == (b & gt).sum() / max(b.sum(), 1) and r[i] == (b & gt).sum() / max(gt.sum(), 1)


def test_tie_rule_has_teeth():
    """On maps whose exact 2 * mean is one of their levels, a correctly rounded mean binarises differently from
    numpy's pairwise one on some maps, and the adaptive F-measure moves: the GPU must sum in numpy's order."""
    rng = np.random.default_rng(3)
    moved = 0
    for shape in ((2, 3), (10, 61), (64, 65)):
        for _ in range(40):
            u, _ = F.tie_map(*shape, rng)
            gt = (rng.random(shape) < 0.4).astype(np.uint8) * 255
            pred, g = M.prepare(u, gt)
            fm = F.cal_adaptive_fm(pred, g)
            assert fm == pytest.approx(_literal_fm(pred, g), abs=1e-12)
            exact_thr = min(2 * (math.fsum(pred.ravel()) / pred.size), 1)
            b = pred >= exact_thr
            i = int(b[g].sum())
            fm_exact = 0.0 if i == 0 else 1.3 * (i / b.sum()) * (i / g.sum()) / (0.3 * (i / b.sum()) + i / g.sum())
            moved += abs(fm - fm_exact) > 1e-6
    assert moved >= 1


def test_get_results_aggregates_over_images():
    rng = np.random.default_rng(4)
    t = F.SODTable()
    rows = []
    for H, W in ((12, 10), (7, 30), (20, 20)):
        pu = rng.integers(0, 256, (H, W)).astype(np.uint8)
        gu = (rng.random((H, W)) < 0.4).astype(np.uint8) * 255
        t.step(pu, gu)
        rows.append(F.table_one(pu, gu))
    r = t.get_results()
    assert r["adpFm"] == pytest.approx(np.mean([x["adp_fm"] for x in rows]), abs=1e-15)
    fm = np.mean([x["fm"] for x in rows], axis=0)
    assert r["maxFm"] == fm.max() and r["meanFm"] == fm.mean()
    assert np.array_equal(r["precision"], np.mean([x["p"] for x in rows], axis=0))
    assert set(r) == {"Smeasure", "wFmeasure", "MAE", "adpEm", "meanEm", "maxEm", "adpFm", "meanFm", "maxFm",
                      "fm_curve", "em_curve", "precision", "recall"}


def test_evaluator_without_images_raises():
    import common
    common.package()
    from dgtd_b200.twig.metric import SODEvaluator
    with pytest.raises(ValueError, match="no image has been processed"):
        SODEvaluator().evaluate()
