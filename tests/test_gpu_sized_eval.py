"""Ground truths of different sizes in one batch: `dgtd_sod_metrics_sized_fwd`, `dgtd_sod_wfm_sized_fwd` and
`dgtd_resize_sigmoid_sized_fwd` (csrc/metric_ops.cu, csrc/stencil_ops.cu) through `PaddedBatch`, the metric
functions, the five evaluators and `cod.forward(mode='predict')`.  The rule under test: image b's values in a sized
call are bit-identical to the uniform entry point on its H_b x W_b crop alone."""
import numpy as np
import pytest
import torch

import common
from oracle import metrics_ref as M
from oracle import wfm_ref as WR

pytestmark = pytest.mark.gpu

# 2 x N, N x 2, 9 x 1000, 384^2, odd sizes, and one image exactly Hmax x Wmax = 384 x 1000
SIZES = [(2, 57), (61, 2), (9, 1000), (384, 384), (33, 47), (384, 1000), (5, 3), (129, 77), (40, 56)]


def _maps(sizes, seed):
    """Per-image (1, H, W) CPU maps: blobs with a noisy prediction, plus the hard cases at fixed positions: empty
    and full ground truth, a tie-heavy point mask and its inverse, and a constant prediction."""
    g = torch.Generator().manual_seed(seed)
    preds, gts = [], []
    for i, (H, W) in enumerate(sizes):
        gt = torch.zeros(1, H, W)
        y0, x0 = int(torch.randint(0, max(1, H // 2), (1,), generator=g)), int(torch.randint(0, max(1, W // 2), (1,), generator=g))
        gt[:, y0:y0 + max(1, H // 2), x0:x0 + max(1, W // 3)] = 1.0
        pred = torch.sigmoid(4 * (gt - 0.5) + 2.0 * torch.randn(1, H, W, generator=g))
        kind = i % 5
        if kind == 1:
            gt.zero_()
        elif kind == 2:
            gt.fill_(1.0)
        elif kind == 3:                              # points on an even grid: many equidistant nearest pixels
            gt.zero_()
            for _ in range(12):
                gt[0, int(torch.randint(0, (H + 1) // 2, (1,), generator=g)) * 2 % H,
                   int(torch.randint(0, (W + 1) // 2, (1,), generator=g)) * 2 % W] = 1.0
            if i % 2:
                gt = 1.0 - gt
            pred = torch.rand(1, H, W, generator=g)
        elif kind == 4:
            pred = torch.full((1, H, W), 0.2)
        preds.append(pred)
        gts.append(gt)
    return preds, gts


def _pkg():
    common.package()
    from dgtd_b200.twig import padded
    from dgtd_b200.twig.metric import sod
    return padded.PaddedBatch, sod


def _sized(preds, gts):
    """(B,2) MAE/S, (B,2,256) curves, (B,) F^w of one sized call per metric, as numpy."""
    _, sod = _pkg()
    p = [x.cuda() for x in preds]
    g = [x.cuda() for x in gts]
    out, cur = sod.sod_metrics(p, g, curves=True)
    wfm = sod.weighted_fmeasure(p, g)
    return out.cpu().numpy(), cur.cpu().numpy(), wfm.cpu().numpy()


def _uniform(pred, gt):
    _, sod = _pkg()
    p, g = pred[None].cuda(), gt[None].cuda()
    out, cur = sod.sod_metrics(p, g, curves=True)
    return out.cpu().numpy()[0], cur.cpu().numpy()[0], sod.weighted_fmeasure(p, g).cpu().numpy()[0]


def test_each_image_equals_the_uniform_call_on_its_crop():
    preds, gts = _maps(SIZES, seed=0)
    out, cur, wfm = _sized(preds, gts)
    assert out.shape == (len(SIZES), 2) and cur.shape == (len(SIZES), 2, 256) and wfm.shape == (len(SIZES),)
    for b in range(len(SIZES)):
        o, c, w = _uniform(preds[b], gts[b])
        assert np.array_equal(out[b], o) and np.array_equal(cur[b], c) and np.array_equal(wfm[b], w), SIZES[b]


def test_sized_call_matches_the_oracle():
    preds, gts = _maps(SIZES, seed=1)
    out, cur, wfm = _sized(preds, gts)
    for b, (p, g) in enumerate(zip(preds, gts)):
        pu, gu = M.quantise(p[None].numpy())[0], M.quantise(g[None].numpy())[0]
        ref = [M.mae_one(pu, gu), M.smeasure_one(pu, gu)]
        assert np.abs(out[b] - ref).max() <= 1e-12, (SIZES[b], out[b], ref)
        assert np.abs(cur[b, 0] - M.fmeasure_curve_one(pu, gu)).max() <= 1e-12, SIZES[b]
        assert np.abs(cur[b, 1] - M.emeasure_curve_one(pu, gu)).max() <= 1e-12, SIZES[b]
        assert abs(wfm[b] - WR.wfm_one(pu, gu)) <= 1e-12, (SIZES[b], wfm[b])


def test_padding_is_never_read():
    PaddedBatch, sod = _pkg()
    preds, gts = _maps(SIZES, seed=2)
    base = _sized(preds, gts)
    for fill in ("nan", "random"):
        p, g = PaddedBatch.from_list([x.cuda() for x in preds]), PaddedBatch.from_list([x.cuda() for x in gts])
        for t in (p.data, g.data):
            pad = torch.full_like(t, float("nan")) if fill == "nan" else torch.rand(t.shape, device="cuda")
            for b, (h, w) in enumerate(p.sizes):
                pad[b, :, :h, :w] = t[b, :, :h, :w]
            t.copy_(pad)
        out, cur = sod.sod_metrics(p, g, curves=True)
        wfm = sod.weighted_fmeasure(p, g)
        for a, e in zip((out, cur, wfm), base):
            assert np.array_equal(a.cpu().numpy(), e), fill


def test_full_sizes_equal_the_uniform_call():
    PaddedBatch, sod = _pkg()
    B, H, W = 5, 70, 91
    preds, gts = _maps([(H, W)] * B, seed=3)
    pred, gt = torch.stack(preds).cuda(), torch.stack(gts).cuda()
    p, g = PaddedBatch(pred, [(H, W)] * B), PaddedBatch(gt, [(H, W)] * B)
    o1, c1 = sod.sod_metrics(p, g, curves=True)
    o0, c0 = sod.sod_metrics(pred, gt, curves=True)
    assert torch.equal(o1, o0) and torch.equal(c1, c0)
    assert torch.equal(sod.weighted_fmeasure(p, g), sod.weighted_fmeasure(pred, gt))


def test_values_do_not_depend_on_the_batch():
    preds, gts = _maps(SIZES, seed=4)
    a = _sized(preds, gts)
    # image 4 (33 x 47) and image 5 (384 x 1000) again, with other neighbours and a larger buffer
    extra_p, extra_g = _maps([(100, 20), (400, 1030)], seed=5)
    b = _sized([extra_p[0], preds[5], extra_p[1], preds[4]], [extra_g[0], gts[5], extra_g[1], gts[4]])
    for i, j in ((5, 1), (4, 3)):
        assert all(np.array_equal(x[i], y[j]) for x, y in zip(a, b)), (i, j)


def test_out_of_range_device_sizes_give_nan():
    """The C entry points check the sizes themselves: an image whose size breaks 2 <= H_b <= Hmax, 2 <= W_b <= Wmax
    reads nothing and gets NaN; the other images are unaffected."""
    from dgtd_b200.twig.ops import capi
    from dgtd_b200.twig.ops.capi import call, ptr, stream
    preds, gts = _maps([(30, 40)] * 4, seed=6)
    pred, gt = torch.stack(preds).cuda(), torch.stack(gts).cuda()
    sizes = torch.tensor([[30, 40], [1, 40], [30, 41], [-3, 5]], dtype=torch.int32, device="cuda")
    lib = capi.load()
    ws = torch.empty(max(int(lib.dgtd_sod_metrics_ws_bytes(4, 30, 40)), int(lib.dgtd_sod_wfm_ws_bytes(4, 30, 40))),
                     device="cuda", dtype=torch.uint8)
    out = torch.empty(4, 2, device="cuda", dtype=torch.float64)
    cur = torch.empty(4, 2, 256, device="cuda", dtype=torch.float64)
    wfm = torch.empty(4, device="cuda", dtype=torch.float64)
    call("dgtd_sod_metrics_sized_fwd", ptr(pred), ptr(gt), ptr(sizes), ptr(ws), ptr(out), ptr(cur), 4, 30, 40, stream())
    call("dgtd_sod_wfm_sized_fwd", ptr(pred), ptr(gt), ptr(sizes), ptr(ws), ptr(wfm), 4, 30, 40, stream())
    prob = torch.empty(4, 1, 30, 40, device="cuda")
    call("dgtd_resize_sigmoid_sized_fwd", ptr(torch.zeros(4, 1, 8, 8, device="cuda")), ptr(prob), ptr(sizes), 4, 8, 8,
         30, 40, stream())
    assert torch.isnan(out[1:]).all() and torch.isnan(cur[1:]).all() and torch.isnan(wfm[1:]).all()
    assert torch.isnan(prob[1:]).all() and torch.equal(prob[0], torch.full_like(prob[0], 0.5))
    o, c, w = _uniform(preds[0], gts[0])
    assert np.array_equal(out[0].cpu().numpy(), o) and np.array_equal(cur[0].cpu().numpy(), c) and wfm[0].item() == w


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_predict_with_labels_of_different_sizes(precision):
    PaddedBatch, _ = _pkg()
    from dgtd_b200.twig.model import hitnet
    from dgtd_b200.twig.model.texture_diffuser import set_precision
    from dgtd_b200.twig.ops.functions import hitnet_func as HF
    from dgtd_b200.twig.ops.functions import texture_diffusion_func as OP
    m = hitnet.cod(binary_thresh=0.2).eval()
    common.hitnet_fixture_params_(m.hitnet, seed=0)
    m = m.cuda()
    set_precision(m, precision)
    B, S = 4, 128
    image, depth = common.synthetic_inputs(B, S, seed=11)
    image, depth = image.cuda(), depth.cuda()
    sizes = [(100, 151), (128, 128), (77, 300), (2, 9)]       # (128, 128) is the x8 grid itself: copied
    g = torch.Generator().manual_seed(12)
    labels = [(torch.rand(1, h, w, generator=g) > 0.5).float() for h, w in sizes]
    prob, lab = m(None, image, labels, depth, mode="predict")
    assert isinstance(prob, PaddedBatch) and isinstance(lab, PaddedBatch)
    assert prob.sizes == lab.sizes == tuple(sizes) and prob.data.shape == lab.data.shape == (B, 1, 128, 300)
    _, out8 = m.hitnet.predict_logits(image, depth, None)
    for b, (h, w) in enumerate(sizes):
        want = HF.sigmoid(OP.resize_nchw(out8[b:b + 1], (h, w)))[0]
        assert torch.equal(prob.unbind()[b], want), (precision, b)
        assert torch.equal(lab.unbind()[b].cpu(), labels[b])
        assert float(prob.data[b, :, h:, :].abs().sum()) == 0 and float(prob.data[b, :, :, w:].abs().sum()) == 0
    with pytest.raises(NotImplementedError):
        m(None, image, labels, depth, mode="tensor")
    set_precision(m, None)


def test_evaluators_take_ragged_batches():
    PaddedBatch, sod = _pkg()
    evs = {"mae": (sod.MAE(), M.RunningMetric(M.mae_one)), "sm": (sod.Smeasure(), M.RunningMetric(M.smeasure_one)),
           "wfm": (sod.WeightedFmeasure(), M.RunningMetric(WR.wfm_one)),
           "fm": (sod.Fmeasure(), M.RunningCurveMetric(M.fmeasure_curve_one)),
           "em": (sod.Emeasure(), M.RunningCurveMetric(M.emeasure_curve_one))}
    records = {k: [] for k in evs}
    batches = [[(31, 45), (64, 20), (9, 70)], [(50, 50), (3, 33)], [(17, 90), (90, 17), (40, 41), (12, 12)]]
    for i, sizes in enumerate(batches):
        preds, gts = _maps(sizes, seed=20 + i)
        as_padded = i % 2 == 0                    # alternate the two accepted forms
        p = PaddedBatch.from_list([x.cuda() for x in preds]) if as_padded else [x.cuda() for x in preds]
        g = PaddedBatch.from_list([x.cuda() for x in gts]) if as_padded else [x.cuda() for x in gts]
        for key, (ev, ref) in evs.items():
            ev.process(None, (p, g))
            for pp, gg in zip(preds, gts):        # the oracle takes one size per call: its record after the batch's
                ref.process(pp[None].numpy(), gg[None].numpy())    # last image is the running value of the batch
            records[key].append(ref.results[-1])
    for key, (ev, _) in evs.items():
        assert [set(r) for r in ev.results] == [{key}] * len(batches)
        got = [r[key] for r in ev.results]
        assert np.abs(np.array(got) - np.array(records[key])).max() <= 1e-12, (key, got, records[key])
        assert abs(list(ev.evaluate().values())[0] - sum(records[key]) / len(records[key])) <= 1e-12


def test_bad_sizes_are_rejected_before_any_launch():
    PaddedBatch, sod = _pkg()
    from dgtd_b200.twig.ops import capi
    a = [torch.rand(1, 10, 12, device="cuda"), torch.rand(1, 7, 9, device="cuda")]
    b = [torch.rand(1, 10, 12, device="cuda"), torch.rand(1, 9, 7, device="cuda")]
    n = capi.launch_count()
    with pytest.raises(ValueError, match="differ"):
        sod.sod_metrics(a, b)
    with pytest.raises(ValueError, match="at least 2"):
        sod.weighted_fmeasure([torch.rand(1, 1, 12, device="cuda")] * 2, [torch.rand(1, 1, 12, device="cuda")] * 2)
    with pytest.raises(ValueError, match="fit the 10 x 12 buffer"):
        PaddedBatch(torch.rand(2, 1, 10, 12, device="cuda"), [(10, 12), (11, 12)])
    assert capi.launch_count() == n
