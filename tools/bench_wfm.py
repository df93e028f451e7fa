"""Weighted F-measure timing (`weighted_fmeasure`, csrc/metric_ops.cu) at the evaluation sizes, the five-evaluator batch
(`sod_metrics(curves=True)` + `weighted_fmeasure`), a per-kernel split, and the host SciPy transcription for scale.

Each size is timed two ways over N launches after warm-up: back to back (the 64 x 384^2 fp32 maps, 75 MB, stay in the
126 MB L2) and one launch at a time with a 512 MB write between launches that evicts L2 (inputs read from HBM)."""
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
from dgtd_b200.twig.metric import sod_metrics, weighted_fmeasure  # noqa: E402
from oracle import metrics_ref as M  # noqa: E402
from oracle import wfm_ref as WR  # noqa: E402

N = 50
# bytes per pixel the passes move: quantise 8 read + 2 written, column pass 1 read + 4 written, row pass 4 + 2 read +
# 1 written, Gaussian pass 3 read (the envelope stacks, the nearest-pixel gathers and the halo re-reads not counted)
BYTES_PER_PIXEL = 8 + 2 + 1 + 4 + 4 + 2 + 1 + 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or f"{torch.cuda.get_device_name(0)}, power limit unknown"


def maps(B, S, seed=0):
    g = torch.Generator().manual_seed(seed)
    gt = torch.zeros(B, 1, S, S)
    for b in range(B):
        for _ in range(2):
            y0, x0 = (int(v) for v in torch.randint(0, S // 2, (2,), generator=g))
            hh, ww = (int(v) for v in torch.randint(S // 16, S // 2, (2,), generator=g))
            gt[b, 0, y0:y0 + hh, x0:x0 + ww] = 1.0
    pred = torch.sigmoid(4 * (gt - 0.5) + 2.0 * torch.randn(B, 1, S, S, generator=g))
    return pred.cuda(), gt.cuda()


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


def main():
    assert torch.cuda.is_available(), "bench_wfm needs a CUDA device"
    print(f"card: {card()}")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    for B, S in ((64, 384), (64, 352), (8, 768)):
        pred, gt = maps(B, S)
        warm, cold = timed(lambda: weighted_fmeasure(pred, gt)), timed(lambda: weighted_fmeasure(pred, gt), flush)
        px = B * S * S
        print(f"weighted_fmeasure B={B} {S}^2: {warm:.4f} ms back to back (L2-warm), {cold:.4f} ms with L2 flushed; "
              f"{BYTES_PER_PIXEL} B/pixel -> {px * BYTES_PER_PIXEL / (cold * 1e6):.0f} GB/s (flushed)")
    pred, gt = maps(64, 384)
    five = lambda: (sod_metrics(pred, gt, curves=True), weighted_fmeasure(pred, gt))  # noqa: E731
    print(f"five evaluators (sod_metrics(curves=True) + weighted_fmeasure) B=64 384^2: {timed(five):.4f} ms back to "
          f"back, {timed(five, flush):.4f} ms with L2 flushed")

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            weighted_fmeasure(pred, gt)
        torch.cuda.synchronize()
    print("per kernel, B=64 384^2 back to back (torch.profiler, mean over 10 calls):")
    for e in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
        if e.device_time_total > 0:
            print(f"  {e.key[:70]:70s} {e.device_time_total / 10 / 1e3:.4f} ms")

    p8, g8 = M.quantise(pred[:2].cpu().numpy()), M.quantise(gt[:2].cpu().numpy())
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from test_oracle_wfm import _scipy_wfm
        import scipy  # noqa: F401
        t = time.perf_counter()
        for p, g in zip(p8, g8):
            _scipy_wfm(p, g)
        print(f"host (CPU) SciPy transcription, 2 images 384^2: {(time.perf_counter() - t) * 1e3:.1f} ms")
    except ImportError:
        print("host (CPU) SciPy transcription: scipy not installed here")
    t = time.perf_counter()
    ref = [WR.wfm_one(p, g) for p, g in zip(p8, g8)]
    print(f"host (CPU) numpy oracle, 2 images 384^2: {(time.perf_counter() - t) * 1e3:.1f} ms; "
          f"max |GPU - oracle| = {np.abs(weighted_fmeasure(pred[:2], gt[:2]).cpu().numpy() - ref).max():.2e}")


if __name__ == "__main__":
    main()
