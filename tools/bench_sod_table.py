"""The whole COD table (`sod_metrics_full`, `SODEvaluator`) against what it replaces.

  (a) `sod_metrics(curves=True)` against `sod_metrics_full` at B = 64, 384^2: the cost of the adaptive values and
      the precision / recall curves;
  (b) `SODEvaluator.process` against the five existing evaluators' `process` (MAE, Smeasure, Fmeasure, Emeasure,
      WeightedFmeasure), on that batch and on the 64 ragged sizes of tools/bench_sized_eval.py.

Each is timed with CUDA events over N calls after warm-up, two ways: back to back (the 64 x 384^2 fp32 maps, 75 MB,
stay in the 126 MB L2) and one call at a time with a 512 MB write between calls that evicts L2.  The old evaluators
synchronise with the host inside `process`; the events include those waits.  A per-kernel split of `sod_metrics_full`
(torch.profiler) follows."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_sized_eval import card, crops, sizes_mix  # noqa: E402
from bench_wfm import maps  # noqa: E402
from dgtd_b200.twig.metric import sod  # noqa: E402
from dgtd_b200.twig.padded import PaddedBatch  # noqa: E402

N = 50


def timed(fn, flush=None):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    if flush is None:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(N):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / N
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(N)]
    for a, b in ev:
        flush.fill_(1)
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / N


def both(fn, flush):
    return f"{timed(fn):.4f} ms back to back (L2-warm), {timed(fn, flush):.4f} ms with L2 flushed"


def main():
    assert torch.cuda.is_available(), "bench_sod_table needs a CUDA device"
    print(f"card: {card()}")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    pred, gt = maps(64, 384)
    vals, cur = sod.sod_metrics_full(pred, gt)
    out, c2 = sod.sod_metrics(pred, gt, curves=True)
    assert torch.equal(vals[:, :2], out) and torch.equal(cur[:, :2], c2)
    print("(a) B=64 384^2, MAE / S / F / E curves of the two calls bit-identical")
    print(f"    sod_metrics(curves=True): {both(lambda: sod.sod_metrics(pred, gt, curves=True), flush)}")
    print(f"    sod_metrics_full:         {both(lambda: sod.sod_metrics_full(pred, gt), flush)}")

    def five(p, g):
        evs = [sod.MAE(), sod.Smeasure(), sod.Fmeasure(), sod.Emeasure(), sod.WeightedFmeasure()]
        return lambda: [e.process(None, (p, g)) for e in evs]

    def table(p, g):
        ev = sod.SODEvaluator()
        return lambda: ev.process(None, (p, g))

    sizes = sizes_mix()
    rp, rg = crops(sizes)
    rp, rg = PaddedBatch.from_list(rp), PaddedBatch.from_list(rg)
    for name, (p, g) in (("B=64 384^2", (pred, gt)), ("64 ragged sizes, buffer %d x %d" % tuple(rp.data.shape[2:]),
                                                      (rp, rg))):
        print(f"(b) process per batch, {name}")
        print(f"    five evaluators: {both(five(p, g), flush)}")
        print(f"    SODEvaluator:    {both(table(p, g), flush)}")
    ev = sod.SODEvaluator()
    ev.process(None, (rp, rg))
    print("    SODEvaluator on the ragged batch:",
          {k: round(v, 6) for k, v in ev.evaluate().items() if not isinstance(v, np.ndarray)})

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            sod.sod_metrics_full(pred, gt)
        torch.cuda.synchronize()
    print("per kernel of sod_metrics_full, B=64 384^2 back to back (torch.profiler, mean over 10 calls):")
    for e in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
        if e.device_time_total > 0:
            print(f"  {e.key[:70]:70s} {e.device_time_total / 10 / 1e3:.4f} ms")


if __name__ == "__main__":
    main()
