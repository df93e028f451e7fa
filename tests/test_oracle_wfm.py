"""The numpy restatement of pysodmetrics' weighted F-measure (oracle/wfm_ref.py::wfm_one) and of its feature
transform (`nearest_foreground`) against SciPy, which the library itself uses, and on hand cases."""
import numpy as np
import pytest

from oracle import metrics_ref as M
from oracle import wfm_ref as WR


def _masks(rng, n):
    """Random densities, rectangles touching the border, even-grid point sets (many equidistant foreground pixels),
    2 x N and N x 2 maps and single pixels; sizes 2..70."""
    out = []
    for t in range(n):
        H, W = (int(v) for v in rng.integers(2, 71, 2))
        kind = t % 5
        if kind == 0:
            m = rng.random((H, W)) < rng.choice([0.005, 0.05, 0.3, 0.8])
        elif kind == 1:
            m = np.zeros((H, W), bool)
            for _ in range(int(rng.integers(1, 4))):
                y0, x0 = int(rng.integers(0, H)), int(rng.integers(0, W))
                m[y0:y0 + int(rng.integers(1, H + 1)), x0:x0 + int(rng.integers(1, W + 1))] = True
            m[int(rng.integers(0, H)), W - 1] = True
        elif kind == 2:
            m = np.zeros((H, W), bool)
            s = int(rng.integers(2, 6))
            for _ in range(int(rng.integers(1, 16))):
                m[int(rng.integers(0, (H + s - 1) // s)) * s, int(rng.integers(0, (W + s - 1) // s)) * s] = True
        elif kind == 3:
            m = rng.random((2, W) if t % 2 else (H, 2)) < 0.3
        else:
            m = np.zeros((H, W), bool)
            m[int(rng.integers(0, H)), int(rng.integers(0, W))] = True
        if m.any():
            out.append(m)
    return out


def test_feature_transform_matches_scipy():
    ndimage = pytest.importorskip("scipy.ndimage")
    masks = _masks(np.random.default_rng(0), 600)
    assert len(masks) >= 500
    for m in masks:
        dst, idx = ndimage.distance_transform_edt(m == 0, return_indices=True)
        d2, r, c = WR.nearest_foreground(m)
        assert np.array_equal(r, idx[0]) and np.array_equal(c, idx[1]), m.shape
        assert np.array_equal(np.sqrt(d2.astype(np.float64)), dst), m.shape


def _gauss2d(shape=(7, 7), sigma=5):
    m, n = [(ss - 1) / 2 for ss in shape]
    y, x = np.ogrid[-m:m + 1, -n:n + 1]
    h = np.exp(-(x * x + y * y) / (2 * sigma * sigma))
    h[h < np.finfo(h.dtype).eps * h.max()] = 0
    sumh = h.sum()
    if sumh != 0:
        h /= sumh
    return h


def _scipy_wfm(pred_u8, gt_u8, beta=1.0):
    """pysodmetrics 1.3.1 `WeightedFmeasure.cal_wfm` transcribed as published."""
    from scipy.ndimage import convolve, distance_transform_edt as bwdist
    pred, gt = M.prepare(pred_u8, gt_u8)
    if np.all(~gt):
        return 0.0
    Dst, Idxt = bwdist(gt == 0, return_indices=True)
    E = np.abs(pred - gt)
    Et = np.copy(E)
    Et[gt == 0] = Et[Idxt[0][gt == 0], Idxt[1][gt == 0]]
    EA = convolve(Et, weights=_gauss2d(), mode="constant", cval=0)
    MIN_E_EA = np.where(gt & (EA < E), EA, E)
    B = np.where(gt == 0, 2 - np.exp(np.log(0.5) / 5 * Dst), np.ones_like(gt))
    Ew = MIN_E_EA * B
    TPw = np.sum(gt) - np.sum(Ew[gt == 1])
    FPw = np.sum(Ew[gt == 0])
    R = 1 - np.mean(Ew[gt == 1])
    P = TPw / (TPw + FPw + M.EPS)
    return (1 + beta) * R * P / (R + beta * P + M.EPS)


def _maps(rng, H, W, kind):
    gt = np.zeros((H, W), np.uint8)
    if kind == "random":
        gt[rng.random((H, W)) < 0.3] = 255
        pred = rng.integers(0, 256, (H, W)).astype(np.uint8)
    else:
        for _ in range(2):
            y0, x0 = int(rng.integers(0, max(1, H // 2))), int(rng.integers(0, max(1, W // 2)))
            gt[y0:y0 + int(rng.integers(1, max(2, H // 2))), x0:x0 + int(rng.integers(1, max(2, W // 2)))] = 255
        p = 1 / (1 + np.exp(-(4 * (gt / 255.0 - 0.5) + 2 * rng.standard_normal((H, W)))))
        pred = (p.astype(np.float32) * np.float32(255)).astype(np.uint8)
    return pred, gt


def test_wfm_matches_the_scipy_transcription():
    pytest.importorskip("scipy.ndimage")
    rng = np.random.default_rng(1)
    cases = [_maps(rng, H, W, kind) for kind in ("random", "blobs") for H, W in ((5, 7), (33, 40), (64, 48), (2, 30),
                                                                                  (30, 2), (96, 80))]
    H, W = 24, 40
    blob = np.zeros((H, W), np.uint8)
    blob[6:18, 10:30] = 255
    cases += [(rng.integers(0, 256, (H, W)).astype(np.uint8), np.full((H, W), 255, np.uint8)),   # full ground truth
              (np.full((H, W), 51, np.uint8), blob),                                            # constant prediction
              (rng.integers(0, 256, (H, W)).astype(np.uint8), np.zeros((H, W), np.uint8))]      # empty ground truth
    for pred, gt in cases:
        want = _scipy_wfm(pred, gt)
        assert abs(WR.wfm_one(pred, gt) - want) <= 1e-12, (pred.shape, WR.wfm_one(pred, gt), want)


def test_hand_cases():
    gt = np.zeros((16, 20), np.uint8)
    gt[4:12, 5:15] = 255                                     # >= 3 px from every border
    assert abs(WR.wfm_one(gt.copy(), gt) - 1.0) < 1e-12       # perfect prediction
    assert abs(WR.wfm_one(255 - gt, gt)) < 1e-12              # inverted prediction: every foreground error is 1
    rng = np.random.default_rng(2)
    assert WR.wfm_one(rng.integers(0, 256, (16, 20)).astype(np.uint8), np.zeros_like(gt)) == 0.0


def _wfm_with_tie_rule(pred_u8, gt_u8, row_first):
    """wfm_one with a brute-force feature transform: among equidistant foreground pixels take the lowest
    (row, column) when `row_first`, else the lowest (column, row)."""
    pred, gt = M.prepare(pred_u8, gt_u8)
    H, W = gt.shape
    fr, fc = np.nonzero(gt)
    yy, xx = np.mgrid[0:H, 0:W]
    d2 = (yy[..., None] - fr) ** 2 + (xx[..., None] - fc) ** 2
    big = 4 * H * W
    key = d2 * big * big + (fr * big + fc if row_first else fc * big + fr)
    k = key.argmin(-1)
    dst = np.sqrt(d2.min(-1).astype(np.float64))
    E = np.abs(pred - gt)
    Et = E[fr[k], fc[k]]
    pad = np.zeros((H + 6, W + 6))
    pad[3:-3, 3:-3] = Et
    K = _gauss2d()
    EA = sum(K[i, j] * pad[i:i + H, j:j + W] for i in range(7) for j in range(7))
    ew = np.where(gt & (EA < E), EA, E) * np.where(gt, 1.0, 2 - np.exp(np.log(0.5) / 5 * dst))
    tpw, fpw = np.sum(gt) - np.sum(ew[gt]), np.sum(ew[~gt])
    R = 1 - np.mean(ew[gt])
    P = tpw / (tpw + fpw + M.EPS)
    return 2 * R * P / (R + P + M.EPS)


def test_tie_rule_moves_the_value():
    """On an even-grid point set most background pixels have several nearest foreground pixels; taking them in
    (row, column) instead of (column, row) order moves F^w by far more than the 1e-12 bar."""
    rng = np.random.default_rng(3)
    H, W = 40, 56
    gt = np.zeros((H, W), np.uint8)
    for _ in range(12):
        gt[int(rng.integers(0, H // 2)) * 2, int(rng.integers(0, W // 2)) * 2] = 255
    pred = rng.integers(0, 256, (H, W)).astype(np.uint8)
    got = WR.wfm_one(pred, gt)
    assert abs(got - _wfm_with_tie_rule(pred, gt, row_first=False)) <= 1e-12
    assert abs(got - _wfm_with_tie_rule(pred, gt, row_first=True)) > 1e-6


def test_running_mean_protocol():
    rng = np.random.default_rng(4)
    m = M.RunningMetric(WR.wfm_one)
    vals = []
    for _ in range(3):
        p = rng.random((2, 1, 12, 10), dtype=np.float32)
        g = (rng.random((2, 1, 12, 10)) > 0.6).astype(np.float32)
        m.process(p, g)
        vals += [WR.wfm_one(a, b) for a, b in zip(M.quantise(p), M.quantise(g))]
    assert abs(m.compute_metrics() - np.mean([np.mean(vals[:2]), np.mean(vals[:4]), np.mean(vals[:6])])) < 1e-15
