"""Dataset preprocessing of decoded RGB-D images on the GPU (`preprocess_rgbd`, csrc/preprocess_ops.cu) against the
reference datasets' host transforms (PIL Resize + ToTensor + Normalize, convert('L') for the depth).

B = 64 seeded source sizes from 250 to 1500 px a side: JPEG-like RGB (a smooth field plus noise) and RGB depth
renderings.  Printed, with the card and its power limit:
  (a) the four kernel launches alone, CUDA events over N calls after warm-up, from a packed buffer already on the
      device;
  (b) the packed host-to-device copy alone, CUDA events over N copies;
  (c) host packing into the pinned staging buffer, host clock;
  (d) the whole call, `preprocess_rgbd` from numpy arrays to device tensors, host clock ending in a synchronise;
  (e) the host torchvision path per image on one core, and over 64 images on all cores of the host (one process
      per core), with the core count (needs PIL and torchvision; reported as not measured without them).
The GPU result is checked bit for bit against oracle/preprocess_ref.py on four images first."""
import multiprocessing as mp
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
from dgtd_b200.twig import preprocess as PP  # noqa: E402
from oracle import preprocess_ref as P  # noqa: E402

N = 50
SIZE = (384, 384)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or f"{torch.cuda.get_device_name(0)}, power limit unknown"


def inputs(n=64, seed=0):
    g = np.random.default_rng(seed)
    rgbs, deps = [], []
    for _ in range(n):
        h, w = int(g.integers(250, 1501)), int(g.integers(250, 1501))
        y, x = np.mgrid[0:h, 0:w]
        for out in (rgbs, deps):
            f = g.uniform(0.003, 0.05, (2, 3))
            base = 127.5 + 110 * np.sin(x[..., None] * f[0] + y[..., None] * f[1] + g.uniform(0, 6, 3))
            out.append(np.clip(base + g.normal(0, 12, (h, w, 3)), 0, 255).astype(np.uint8))
    return rgbs, deps


def events_ms(fn, n=N):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def host_ms(fn, n):
    fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / n


def _tv_one(args):
    """The reference dataset's transforms of one RGB-D pair on the host."""
    from PIL import Image
    import torchvision.transforms as T
    rgb, dep = args
    a = T.Compose([T.Resize(SIZE), T.ToTensor(), T.Normalize(P.IMAGENET_MEAN, P.IMAGENET_STD)])(Image.fromarray(rgb))
    b = T.Compose([T.Resize(SIZE), T.ToTensor()])(Image.fromarray(dep).convert("L"))
    return a.shape[0] + b.shape[0]


def _init_worker():
    torch.set_num_threads(1)


def main():
    assert torch.cuda.is_available(), "bench_preprocess needs a CUDA device"
    print(f"card: {card()}")
    rgbs, deps = inputs()
    B = len(rgbs)
    mpx = sum(r.shape[0] * r.shape[1] for r in rgbs) / 1e6
    desc, total = PP._layout(rgbs, deps)
    print(f"B = {B}: sizes {min(min(r.shape[:2]) for r in rgbs)} to {max(max(r.shape[:2]) for r in rgbs)} px a side, "
          f"{mpx:.1f} Mpx of RGB plus RGB depth renderings; packed buffer {total / 1e6:.1f} MB; output "
          f"{B * 4 * SIZE[0] * SIZE[1] * 4 / 1e6:.1f} MB fp32")

    img, dep = PP.preprocess_rgbd(rgbs, deps, size=SIZE)
    want = [(P.preprocess_rgb(rgbs[b], SIZE), P.preprocess_depth(deps[b], SIZE)) for b in (0, 1, 31, 63)]
    for (wi, wd), b in zip(want, (0, 1, 31, 63)):
        assert np.array_equal(img[b].cpu().numpy(), wi) and np.array_equal(dep[b].cpu().numpy(), wd), b
    print("GPU result equals the oracle bit for bit on images 0, 1, 31, 63")

    host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    view = host.numpy()
    tc = host_ms(lambda: PP._fill(view, desc, rgbs, deps), 10)
    packed = torch.empty(total, dtype=torch.uint8, device="cuda")
    tb = events_ms(lambda: packed.copy_(host, non_blocking=True))
    m32, s32 = np.asarray(P.IMAGENET_MEAN, np.float32), np.asarray(P.IMAGENET_STD, np.float32)
    ta = events_ms(lambda: PP._launch(packed, host, desc, SIZE, m32, s32))
    td = host_ms(lambda: PP.preprocess_rgbd(rgbs, deps, size=SIZE), 10)
    print(f"(a) kernels (plan, coef, pass1, pass2): {ta:.3f} ms per batch of {B} "
          f"({total / ta / 1e6:.0f} GB/s packed in + {B * 4 * SIZE[0] * SIZE[1] * 4 / ta / 1e6:.0f} GB/s out)")
    print(f"(b) packed host-to-device copy: {tb:.3f} ms ({total / tb / 1e6:.1f} GB/s)")
    print(f"(c) host packing into pinned memory: {tc:.2f} ms")
    print(f"(d) whole preprocess_rgbd call: {td:.2f} ms per batch of {B} ({td / B * 1e3:.0f} us per image)")

    try:
        import PIL  # noqa: F401
        import torchvision  # noqa: F401
    except ImportError:
        print("(e) host torchvision path: not measured (PIL or torchvision is not installed here)")
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    torch.set_num_threads(1)
    pairs = list(zip(rgbs, deps))
    _tv_one(pairs[0])
    t = time.perf_counter()
    for p in pairs[:16]:
        _tv_one(p)
    one = (time.perf_counter() - t) * 1e3 / 16
    with mp.get_context("spawn").Pool(cores, initializer=_init_worker) as pool:
        pool.map(_tv_one, pairs[:cores])
        t = time.perf_counter()
        pool.map(_tv_one, pairs, chunksize=1)
        allc = (time.perf_counter() - t) * 1e3
    print(f"(e) host torchvision path: {one:.2f} ms per image on one core (16 images); {allc:.1f} ms for {B} images "
          f"on {cores} cores ({allc / B:.2f} ms per image)")


if __name__ == "__main__":
    main()
