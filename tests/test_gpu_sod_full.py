"""The whole COD table on the GPU: `sod_metrics_full` (`dgtd_sod_metrics_full_fwd` / `_sized_fwd`, csrc/metric_ops.cu)
against the numpy restatement of pysodmetrics (oracle/sod_full_ref.py), against `sod_metrics(curves=True)` bit for
bit, on maps whose adaptive threshold lands on a prediction level, and `SODEvaluator` against `get_results()`."""
import numpy as np
import pytest
import torch

import common
from oracle import metrics_ref as M
from oracle import sod_full_ref as F

pytestmark = pytest.mark.gpu


def _sod():
    common.package()
    from dgtd_b200.twig.metric import sod
    return sod


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


def _from_u8(u):
    """fp32 maps that the wrappers' `(x * 255).astype(np.uint8)` turns back into u exactly."""
    x = torch.from_numpy((u.astype(np.float32) + np.float32(0.5)) / np.float32(255))
    return torch.where(torch.from_numpy(u == 255), torch.ones_like(x), x)


def _oracle(pred, gt):
    """per image: (adaptive F, adaptive E), precision, recall of the oracle, from fp32 maps (1, H, W)."""
    out = []
    for p, g in zip(pred, gt):
        pu, gu = M.quantise(p[None].numpy())[0], M.quantise(g[None].numpy())[0]
        pp, gg = M.prepare(pu, gu)
        pr, rc = F.cal_pr(pp, gg)
        out.append((np.array([F.cal_adaptive_fm(pp, gg), F.cal_adaptive_em(pp, gg)]), pr, rc))
    return out


def _check_against_oracle(pred, gt, vals, cur):
    for b, (adp, pr, rc) in enumerate(_oracle(pred, gt)):
        assert np.abs(vals[b, 2:] - adp).max() <= 1e-12, (b, vals[b, 2:], adp)
        assert np.abs(cur[b, 2] - pr).max() <= 1e-12 and np.abs(cur[b, 3] - rc).max() <= 1e-12, b


def _full(pred, gt):
    vals, cur = _sod().sod_metrics_full(pred, gt)
    return vals.cpu().numpy(), cur.cpu().numpy()


@pytest.mark.parametrize("shape", [(3, 64, 48), (2, 384, 384), (5, 37, 53), (1, 9, 1000), (2, 2, 300), (4, 2, 3),
                                   (2, 129, 65)])
def test_matches_the_oracle_and_sod_metrics(shape):
    B, H, W = shape
    pred, gt = _blobs(B, H, W, seed=H * W)
    vals, cur = _full(pred.cuda(), gt.cuda())
    assert vals.shape == (B, 4) and cur.shape == (B, 4, 256)
    _check_against_oracle(pred, gt, vals, cur)
    out, c2 = _sod().sod_metrics(pred.cuda(), gt.cuda(), curves=True)
    assert np.array_equal(vals[:, :2], out.cpu().numpy()) and np.array_equal(cur[:, :2], c2.cpu().numpy())


def test_edge_cases():
    """Empty and full ground truth, perfect and inverted predictions, constant 0 (threshold 0: every pixel is
    foreground), constant non-zero (left un-normalised: no pixel reaches 2 * mean) and constant 1 predictions, and
    narrow prediction ranges."""
    H, W = 40, 56
    g = torch.Generator().manual_seed(0)
    blob = torch.zeros(1, 1, H, W)
    blob[..., 6:30, 10:40] = 1.0
    rnd = lambda: torch.rand(1, 1, H, W, generator=g)  # noqa: E731
    full = lambda v: torch.full((1, 1, H, W), v)  # noqa: E731
    cases = [(rnd(), full(0.0)), (rnd(), full(1.0)), (blob.clone(), blob), (1 - blob, blob), (full(0.0), blob),
             (full(0.2), blob), (full(1.0), blob), (full(0.0), full(0.0)), (0.3 + 0.05 * rnd(), blob),
             (0.9 + 0.02 * rnd(), 1 - blob)]
    pred, gt = torch.cat([c[0] for c in cases]), torch.cat([c[1] for c in cases])
    vals, cur = _full(pred.cuda(), gt.cuda())
    _check_against_oracle(pred, gt, vals, cur)
    assert abs(vals[2, 2] - 1.0) < 1e-12 and vals[3, 2] == 0.0 and vals[5, 2] == 0.0 and vals[7, 2:].tolist() == [0, 0]
    assert vals[4, 2] == vals[6, 2] > 0.0


@pytest.mark.parametrize("shape", [(2, 3), (10, 61), (3, 43), (64, 65), (96, 80), (1000, 1000)])
def test_tie_maps_binarise_like_numpy(shape):
    """Maps whose exact 2 * mean is one of their levels, and shuffled arrangements of the same pixels: numpy's rounding
    of the mean decides whether the pixels at that level are foreground, and the GPU must decide the same way."""
    rng = np.random.default_rng(sum(shape))
    n_maps, n_shuffles = (2, 3) if shape == (1000, 1000) else (8, 4)
    preds, gts, maps, decisions = [], [], [], set()
    for _ in range(n_maps):
        u, a = F.tie_map(*shape, rng)
        gu = (rng.random(shape) < 0.4).astype(np.uint8) * 255
        for _ in range(n_shuffles):
            perm = rng.permutation(u.size)
            us, gs = u.ravel()[perm].reshape(shape), gu.ravel()[perm].reshape(shape)
            pp, _ = M.prepare(us, gs)
            decisions.add((a, bool(a / 255 >= F.adaptive_threshold(pp))))
            maps.append(us)
            preds.append(_from_u8(us)[None])
            gts.append(torch.from_numpy(gs.astype(np.float32) / 255)[None])
    pred, gt = torch.stack(preds), torch.stack(gts)
    assert np.array_equal(M.quantise(pred.numpy()), np.stack(maps))
    vals, cur = _full(pred.cuda(), gt.cuda())
    _check_against_oracle(pred, gt, vals, cur)
    if shape in ((10, 61), (64, 65)):
        assert len(decisions) > len({a for a, _ in decisions}), "no map here is decided both ways: the test has no teeth"


def _ragged(sizes, seed):
    g = torch.Generator().manual_seed(seed)
    preds, gts = [], []
    for i, (H, W) in enumerate(sizes):
        gt = torch.zeros(1, H, W)
        gt[:, H // 4:H // 4 + max(1, H // 2), W // 5:W // 5 + max(1, W // 3)] = 1.0
        pred = torch.sigmoid(4 * (gt - 0.5) + 2.0 * torch.randn(1, H, W, generator=g))
        if i % 4 == 1:
            gt.zero_()
        elif i % 4 == 2:
            pred = torch.full((1, H, W), 0.2)
        preds.append(pred)
        gts.append(gt)
    return preds, gts


SIZES = [(2, 57), (61, 2), (9, 1000), (384, 384), (33, 47), (384, 1000), (5, 3), (129, 77), (2, 2), (300, 7)]


def test_sized_call_equals_the_uniform_call_on_each_crop():
    sod = _sod()
    preds, gts = _ragged(SIZES, seed=1)
    vals, cur = _full([p.cuda() for p in preds], [g.cuda() for g in gts])
    for b, (p, g) in enumerate(zip(preds, gts)):
        v1, c1 = _full(p[None].cuda(), g[None].cuda())
        assert np.array_equal(vals[b], v1[0]) and np.array_equal(cur[b], c1[0]), SIZES[b]
    _check_against_oracle(preds, gts, vals, cur)
    from dgtd_b200.twig.padded import PaddedBatch
    for fill in ("nan", "random"):
        p, g = PaddedBatch.from_list([x.cuda() for x in preds]), PaddedBatch.from_list([x.cuda() for x in gts])
        for t in (p.data, g.data):
            pad = torch.full_like(t, float("nan")) if fill == "nan" else torch.rand(t.shape, device="cuda")
            for b, (h, w) in enumerate(p.sizes):
                pad[b, :, :h, :w] = t[b, :, :h, :w]
            t.copy_(pad)
        v2, c2 = sod.sod_metrics_full(p, g)
        assert np.array_equal(v2.cpu().numpy(), vals) and np.array_equal(c2.cpu().numpy(), cur), fill


def test_results_do_not_depend_on_the_batch():
    preds, gts = _ragged(SIZES, seed=2)
    a = _full([p.cuda() for p in preds], [g.cuda() for g in gts])
    extra_p, extra_g = _ragged([(100, 20), (400, 1030)], seed=3)
    b = _full([extra_p[0].cuda(), preds[5].cuda(), extra_p[1].cuda(), preds[4].cuda()],
              [extra_g[0].cuda(), gts[5].cuda(), extra_g[1].cuda(), gts[4].cuda()])
    for i, j in ((5, 1), (4, 3)):
        assert np.array_equal(a[0][i], b[0][j]) and np.array_equal(a[1][i], b[1][j]), (i, j)
    pred, gt = _blobs(4, 96, 80, seed=4)
    whole = _full(pred.cuda(), gt.cuda())
    for i in range(4):
        one = _full(pred[i:i + 1].cuda(), gt[i:i + 1].cuda())
        assert np.array_equal(whole[0][i], one[0][0]) and np.array_equal(whole[1][i], one[1][0])


def test_out_of_range_device_sizes_give_nan():
    _sod()
    from dgtd_b200.twig.ops import capi
    from dgtd_b200.twig.ops.capi import call, ptr, stream
    preds, gts = _ragged([(30, 40)] * 4, seed=5)
    pred, gt = torch.stack(preds).cuda(), torch.stack(gts).cuda()
    sizes = torch.tensor([[30, 40], [1, 40], [30, 41], [-3, 5]], dtype=torch.int32, device="cuda")
    ws = torch.empty(int(capi.load().dgtd_sod_metrics_full_ws_bytes(4, 30, 40)), device="cuda", dtype=torch.uint8)
    vals = torch.empty(4, 4, device="cuda", dtype=torch.float64)
    cur = torch.empty(4, 4, 256, device="cuda", dtype=torch.float64)
    call("dgtd_sod_metrics_full_sized_fwd", ptr(pred), ptr(gt), ptr(sizes), ptr(ws), ptr(vals), ptr(cur), 4, 30, 40,
         stream())
    assert torch.isnan(vals[1:]).all() and torch.isnan(cur[1:]).all()
    v0, c0 = _full(pred[:1], gt[:1])
    assert np.array_equal(vals[0].cpu().numpy(), v0[0]) and np.array_equal(cur[0].cpu().numpy(), c0[0])


def test_evaluator_matches_get_results():
    """Uniform batches (tensors) and ragged ones (PaddedBatch and lists) of unequal lengths: the aggregate is over
    images, not over per-batch records."""
    sod = _sod()
    from dgtd_b200.twig.padded import PaddedBatch
    ev, ref = sod.SODEvaluator(), F.SODTable()
    batches = [("tensor", _blobs(3, 64, 48, seed=10)), ("padded", _ragged([(31, 45), (64, 20), (9, 70)], seed=11)),
               ("tensor", _blobs(1, 40, 40, seed=12)), ("list", _ragged([(50, 50), (3, 33), (17, 90), (90, 17)], 13))]
    for kind, (pred, gt) in batches:
        if kind == "tensor":
            ev.process(None, (pred.cuda(), gt.cuda()))
        elif kind == "padded":
            ev.process(None, (PaddedBatch.from_list([x.cuda() for x in pred]),
                              PaddedBatch.from_list([x.cuda() for x in gt])))
        else:
            ev.process(None, ([x.cuda() for x in pred], [x.cuda() for x in gt]))
        for p, g in zip(pred, gt):
            ref.step(M.quantise(p[None].numpy())[0], M.quantise(g[None].numpy())[0])
    got, want = ev.evaluate(), ref.get_results()
    assert set(got) == set(want)
    for k in want:
        assert np.abs(np.asarray(got[k]) - np.asarray(want[k])).max() <= 1e-12, (k, got[k], want[k])


def test_evaluator_process_does_not_synchronise():
    sod = _sod()
    pred, gt = _blobs(3, 40, 30, seed=20)
    pred, gt = pred.cuda(), gt.cuda()
    ev = sod.SODEvaluator()
    ev.process(None, (pred, gt))                              # the first call loads the library
    torch.cuda.set_sync_debug_mode("error")
    try:
        ev.process(None, (pred, gt))
        ev.process(None, ([p[:, :20 + i] for i, p in enumerate(pred)], [g[:, :20 + i] for i, g in enumerate(gt)]))
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert ev._count == 9 and np.isfinite(ev.evaluate()["adpFm"])


def test_bad_inputs_are_rejected_before_any_launch():
    sod = _sod()
    from dgtd_b200.twig.ops import capi
    from dgtd_b200.twig.padded import PaddedBatch
    a = [torch.rand(1, 10, 12, device="cuda"), torch.rand(1, 7, 9, device="cuda")]
    b = [torch.rand(1, 10, 12, device="cuda"), torch.rand(1, 9, 7, device="cuda")]
    n = capi.launch_count()
    with pytest.raises(ValueError, match="prediction sizes .* differ"):
        sod.sod_metrics_full(a, b)
    with pytest.raises(ValueError, match="prediction buffer .* differs"):
        sod.sod_metrics_full(PaddedBatch(torch.rand(2, 1, 10, 12, device="cuda"), [(10, 12), (7, 9)]),
                             PaddedBatch(torch.rand(2, 1, 10, 13, device="cuda"), [(10, 12), (7, 9)]))
    with pytest.raises(ValueError, match="at least 2"):
        sod.sod_metrics_full([torch.rand(1, 1, 12, device="cuda")] * 2, [torch.rand(1, 1, 12, device="cuda")] * 2)
    with pytest.raises(ValueError, match="at least 2"):
        sod.SODEvaluator().process(None, ([torch.rand(1, 12, 1, device="cuda")], [torch.rand(1, 12, 1, device="cuda")]))
    assert capi.launch_count() == n
    x = torch.rand(1, 1, 1, 40, device="cuda")
    with pytest.raises(RuntimeError, match=r"dgtd_sod_metrics_full_fwd failed \(-1\): sod_metrics_full: bad shape"):
        sod.sod_metrics_full(x, x)
