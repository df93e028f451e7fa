"""Scoring ground truths of different sizes (twig/padded.py, the sized entry points of csrc/metric_ops.cu and
csrc/stencil_ops.cu) against the per-image loop that one shape per batch forces.

On a seeded mix of 64 sizes between 240 and 1024 px a side, portrait and landscape:
  (a) a per-image loop over the five evaluators' entry points (MAE, S-measure, F-measure, E-measure, F^w) on
      contiguous crops, as batch-1 scoring runs them;
  (b) the same five entry points, one sized call each on the padded batch; (a) and (b) must agree bit for bit;
  (c) end to end: `cod.forward(mode='predict')` at B = 64, 384^2 input, bf16, with the ragged labels, then the five
      evaluators' `process`, against 64 batch-1 predicts each followed by the five `process` calls.
(a) and (b) are timed with CUDA events around N repetitions after warm-up, inputs L2-warm (the padded batch is
about 270 MB per map, so most of it comes from HBM).  (c) is timed with a host clock around whole passes, which end
in the evaluators' device-to-host copies."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import common  # noqa: E402

common.package()
from dgtd_b200.twig.metric import sod  # noqa: E402
from dgtd_b200.twig.padded import PaddedBatch  # noqa: E402

N = 10


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or f"{torch.cuda.get_device_name(0)}, power limit unknown"


def sizes_mix(n=64, seed=0):
    g = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        long = int(g.integers(480, 1025))
        short = int(g.integers(240, long + 1))
        out.append((long, short) if g.random() < 0.5 else (short, long))
    return out


def crops(sizes, seed=0):
    g = torch.Generator().manual_seed(seed)
    preds, gts = [], []
    for H, W in sizes:
        gt = torch.zeros(1, H, W)
        for _ in range(2):
            y0, x0 = int(torch.randint(0, H // 2, (1,), generator=g)), int(torch.randint(0, W // 2, (1,), generator=g))
            gt[:, y0:y0 + H // 3, x0:x0 + W // 3] = 1.0
        preds.append(torch.sigmoid(4 * (gt - 0.5) + 2.0 * torch.randn(1, H, W, generator=g)).cuda())
        gts.append(gt.cuda())
    return preds, gts


def five(p, g):
    """What the five evaluators launch: MAE, S-measure, F-measure, E-measure, F^w, each its own entry point."""
    return (sod.sod_metrics(p, g), sod.sod_metrics(p, g), sod.sod_metrics(p, g, curves=True),
            sod.sod_metrics(p, g, curves=True), sod.weighted_fmeasure(p, g))


def event_ms(fn):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(N):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / N


def host_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / reps


def evaluators():
    return [sod.MAE(), sod.Smeasure(), sod.Fmeasure(), sod.Emeasure(), sod.WeightedFmeasure()]


def main():
    assert torch.cuda.is_available(), "bench_sized_eval needs a CUDA device"
    print(f"card: {card()}")
    sizes = sizes_mix()
    preds, gts = crops(sizes)
    p, g = PaddedBatch.from_list(preds), PaddedBatch.from_list(gts)
    real = sum(h * w for h, w in sizes)
    B, _, Hmax, Wmax = p.data.shape
    print(f"64 sizes from {min(min(s) for s in sizes)} to {max(max(s) for s in sizes)} px a side, "
          f"{sum(h > w for h, w in sizes)} portrait; buffer {Hmax} x {Wmax}, {real / 1e6:.1f} Mpx of images in "
          f"{B * Hmax * Wmax / 1e6:.1f} Mpx of buffer ({100 * (1 - real / (B * Hmax * Wmax)):.0f} % padding)")

    loop = lambda: [five(pp[None], gg[None]) for pp, gg in zip(preds, gts)]  # noqa: E731
    sized = lambda: five(p, g)  # noqa: E731
    a, b = loop(), sized()
    names = ("MAE / S", "MAE / S", "F / E curves", "F / E curves", "F^w")
    for k in range(5):
        got = b[k] if k < 2 or k == 4 else b[k][1]
        want = torch.cat([r[k] if k < 2 or k == 4 else r[k][1] for r in a])
        assert torch.equal(got, want), names[k]
        if k in (2, 3):
            assert torch.equal(b[k][0], torch.cat([r[k][0] for r in a]))
    print("(a) and (b) agree bit for bit: per-image MAE, S-measure, F and E curves, F^w")
    ta, tb = event_ms(loop), event_ms(sized)
    print(f"(a) per-image loop, 64 x 5 entry points on crops: {ta:.3f} ms")
    print(f"(b) one sized call per entry point on the padded batch: {tb:.3f} ms ({ta / tb:.1f}x)")

    from dgtd_b200.twig.model import hitnet
    from dgtd_b200.twig.model.texture_diffuser import set_precision
    m = hitnet.cod(binary_thresh=0.2).eval()
    common.hitnet_fixture_params_(m.hitnet, seed=0)
    m = m.cuda()
    set_precision(m, "bf16")
    image, depth = common.synthetic_inputs(64, 384, seed=1)
    image, depth = image.cuda(), depth.cuda()
    labels = gts

    def batched():
        evs = evaluators()
        prob, lab = m(None, image, labels, depth, mode="predict")
        for ev in evs:
            ev.process(None, (prob, lab))
        return [ev.evaluate() for ev in evs]

    def batch1():
        evs = evaluators()
        for i in range(64):
            prob, lab = m(None, image[i:i + 1], [labels[i]], depth[i:i + 1], mode="predict")
            for ev in evs:
                ev.process(None, (prob, lab))
        return [ev.evaluate() for ev in evs]

    with torch.no_grad():
        rb, r1 = batched(), batch1()
        tc, t1 = host_ms(batched, 5), host_ms(batch1, 2)
    diff = max(abs(list(x.values())[0] - list(y.values())[0]) for x, y in zip(rb, r1))
    print(f"(c) predict B=64 384^2 bf16 + five evaluators, ragged labels: {tc:.1f} ms per 64 images; batch-1 loop: "
          f"{t1:.1f} ms ({t1 / tc:.1f}x); max |difference| of the five scores between the routes {diff:.2e}")
    print("   scores:", {k: round(v, 6) for r in rb for k, v in r.items()})


if __name__ == "__main__":
    main()
