"""Weighted F-measure kernels (csrc/metric_ops.cu, `dgtd_sod_wfm_fwd`) against the numpy restatement of pysodmetrics
(oracle/wfm_ref.py::wfm_one), and the evaluator's running-mean protocol."""
import os

import numpy as np
import pytest
import torch

import common
from oracle import metrics_ref as M
from oracle import wfm_ref as WR

pytestmark = pytest.mark.gpu


def _blobs(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    gt = torch.zeros(B, 1, H, W)
    for b in range(B):
        for _ in range(2):
            y0, x0 = int(torch.randint(0, max(1, H // 2), (1,), generator=g)), int(torch.randint(0, max(1, W // 2), (1,), generator=g))
            hh, ww = int(torch.randint(1, max(2, H // 2), (1,), generator=g)), int(torch.randint(1, max(2, W // 2), (1,), generator=g))
            gt[b, 0, y0:y0 + hh, x0:x0 + ww] = 1.0
    pred = torch.sigmoid(4 * (gt - 0.5) + 2.0 * torch.randn(B, 1, H, W, generator=g))
    return pred, gt


def _oracle(pred, gt):
    return np.array([WR.wfm_one(p, g) for p, g in zip(M.quantise(pred.numpy()), M.quantise(gt.numpy()))])


def _wfm(pred, gt):
    common.package()
    from dgtd_b200.twig.metric import weighted_fmeasure
    return weighted_fmeasure(pred.cuda(), gt.cuda()).cpu().numpy()


@pytest.mark.parametrize("shape", [(3, 64, 48), (2, 384, 384), (2, 352, 352), (5, 37, 53), (1, 9, 1000), (2, 2, 300)])
def test_wfm_matches_the_oracle(shape):
    B, H, W = shape
    pred, gt = _blobs(B, H, W, seed=H + W)
    got, ref = _wfm(pred, gt), _oracle(pred, gt)
    assert got.shape == (B,) and np.abs(got - ref).max() <= 1e-12, (got, ref)


def test_edge_cases_and_ties():
    """Perfect / inverted / constant predictions, empty and full ground truth, and even-grid point masks with random
    predictions, where most background pixels have several nearest foreground pixels."""
    H, W = 40, 56
    g = torch.Generator().manual_seed(0)
    blob = torch.zeros(1, 1, H, W)
    blob[..., 6:30, 10:40] = 1.0
    rnd = lambda: torch.rand(1, 1, H, W, generator=g)  # noqa: E731
    cases = [(blob.clone(), blob), (1 - blob, blob), (torch.full((1, 1, H, W), 0.2), blob),
             (rnd(), torch.zeros(1, 1, H, W)), (rnd(), torch.ones(1, 1, H, W))]
    for step in (2, 3, 4):
        pts = torch.zeros(1, 1, H, W)
        for _ in range(12):
            pts[0, 0, int(torch.randint(0, H // step, (1,), generator=g)) * step,
                int(torch.randint(0, W // step, (1,), generator=g)) * step] = 1.0
        cases += [(rnd(), pts), (rnd(), 1 - pts)]
    pred = torch.cat([c[0] for c in cases])
    gt = torch.cat([c[1] for c in cases])
    got, ref = _wfm(pred, gt), _oracle(pred, gt)
    assert np.abs(got - ref).max() <= 1e-12, (got, ref)
    assert abs(got[0] - 1.0) < 1e-12 and abs(got[1]) < 1e-12 and got[3] == 0.0


@pytest.mark.parametrize("name", ["hitnet_128.npz", "hitnet_352.npz"])
def test_wfm_on_the_reference_probability_maps(name):
    """sigmoid of the reference's golden logits against a fixed blob label and against its own 0.5 mask."""
    golden = np.load(os.path.join(common.GOLDEN, name))
    logits = torch.from_numpy(golden["logits"])
    prob = torch.sigmoid(logits).float()
    B, _, H, W = prob.shape
    mask = np.unpackbits(golden["mask50"])[:logits.numel()].reshape(logits.shape).astype(np.float32)
    blob = torch.zeros(B, 1, H, W)
    blob[..., H // 4:3 * H // 4, W // 5:3 * W // 5] = 1.0
    for gt in (blob, torch.from_numpy(mask)):
        got, ref = _wfm(prob, gt), _oracle(prob, gt)
        assert np.abs(got - ref).max() <= 1e-12, (got, ref)


def test_bit_stable_across_batch_composition():
    pred, gt = _blobs(4, 96, 80, seed=3)
    a = _wfm(pred, gt)
    b = np.concatenate([_wfm(pred[i:i + 1], gt[i:i + 1]) for i in range(4)])
    assert np.array_equal(a, b)


def test_evaluator_follows_the_reference_protocol():
    common.package()
    from dgtd_b200.twig.metric import WeightedFmeasure
    wfm, owfm = WeightedFmeasure(), M.RunningMetric(WR.wfm_one)
    for seed in range(3):
        pred, gt = _blobs(2, 32, 32, seed)
        wfm.process(None, (pred.cuda(), gt.cuda()))
        owfm.process(pred.numpy(), gt.numpy())
    assert abs(wfm.evaluate()["WeightedFmeasure"] - owfm.compute_metrics()) < 1e-12
    assert [set(r) for r in wfm.results] == [{"wfm"}] * 3


@pytest.mark.parametrize("shape", [(1, 1, 1, 40), (1, 1, 40, 1)])
def test_single_row_or_column_is_rejected(shape):
    common.package()
    from dgtd_b200.twig.metric import weighted_fmeasure
    x = torch.rand(*shape, device="cuda")
    with pytest.raises(RuntimeError, match=r"dgtd_sod_wfm_fwd failed \(-1\): sod_wfm: bad shape"):
        weighted_fmeasure(x, x)
