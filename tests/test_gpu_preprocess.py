"""`preprocess_rgbd` (twig/preprocess.py, csrc/preprocess_ops.cu) against oracle/preprocess_ref.py and, where they
are importable, PIL and torchvision themselves.  Every comparison is bit identity."""
import numpy as np
import pytest
import torch

import common
from oracle import preprocess_ref as P

pytestmark = pytest.mark.gpu

# down/down, up/up, mixed, one axis unchanged, identity, 1 x N / N x 1 / 1 x 1, both sides of the pass-order rule
# (vertical first iff H > 100 W and the output is shorter than H), odd sizes and a 4000 x 3000 photo
RAGGED = [(1024, 768), (768, 1024), (200, 300), (5, 7), (250, 1500), (1500, 250), (384, 1000), (1000, 384),
          (384, 200), (200, 384), (384, 384), (1, 50), (50, 1), (1, 1), (1, 1000), (1000, 1), (383, 385),
          (800, 8), (801, 8), (3000, 30), (3001, 30), (1000, 8), (2500, 24), (1400, 13), (250, 2), (380, 3),
          (4000, 3000)]


def _pp():
    common.package()
    from dgtd_b200.twig import preprocess
    return preprocess.preprocess_rgbd


def _image(h, w, c, g):
    """JPEG-like content: a smooth field plus noise, as uint8 (H, W, c)."""
    y, x = np.mgrid[0:h, 0:w]
    f = g.uniform(0.003, 0.05, (2, c))
    base = 127.5 + 110 * np.sin(x[..., None] * f[0] + y[..., None] * f[1] + g.uniform(0, 6, c))
    return np.clip(base + g.normal(0, 12, (h, w, c)), 0, 255).astype(np.uint8)


def _batch(sizes, seed):
    """RGB at each size; depth alternately 3-channel (a colour rendering) and 1-channel, every third one at another
    size than its RGB."""
    g = np.random.default_rng(seed)
    rgbs, deps = [], []
    for i, (h, w) in enumerate(sizes):
        rgbs.append(_image(h, w, 3, g))
        dh, dw = (max(1, h // 2 + 3), max(1, (w * 3) // 4)) if i % 3 == 2 else (h, w)
        d = _image(dh, dw, 3, g)
        deps.append(d if i % 2 == 0 else np.ascontiguousarray(d[..., 0]))
    return rgbs, deps


def _oracle(rgbs, deps, size, mean=P.IMAGENET_MEAN, std=P.IMAGENET_STD):
    return (np.stack([P.preprocess_rgb(r, size, mean, std) for r in rgbs]),
            np.stack([P.preprocess_depth(d, size) for d in deps]))


def _check(got, want):
    img, dep = (t.cpu().numpy() for t in got)
    assert img.dtype == np.float32 and dep.dtype == np.float32
    assert got[0].is_contiguous() and got[1].is_contiguous()
    for b in range(len(want[0])):
        assert np.array_equal(img[b], want[0][b]), f"image {b}: {(img[b] != want[0][b]).sum()} values differ"
        assert np.array_equal(dep[b], want[1][b]), f"depth {b}: {(dep[b] != want[1][b]).sum()} values differ"


@pytest.mark.parametrize("size", [(384, 384), (352, 352), (768, 768)], ids=lambda s: f"{s[0]}")
def test_ragged_batch_equals_oracle(size):
    pp = _pp()
    rgbs, deps = _batch(RAGGED, seed=size[0])
    got = pp(rgbs, deps, size=size)
    _check(got, _oracle(rgbs, deps, size))


def test_ragged_batch_equals_pil_and_torchvision():
    Image = pytest.importorskip("PIL.Image")
    T = pytest.importorskip("torchvision.transforms")
    pp = _pp()
    size = (384, 384)
    rgbs, deps = _batch(RAGGED, seed=7)
    img, dep = pp([torch.from_numpy(r) for r in rgbs], deps, size=size)     # CPU tensors are taken too
    rgb_tf = T.Compose([T.Resize(size), T.ToTensor(), T.Normalize(P.IMAGENET_MEAN, P.IMAGENET_STD)])
    dep_tf = T.Compose([T.Resize(size), T.ToTensor()])
    assert torch.equal(img.cpu(), torch.stack([rgb_tf(Image.fromarray(r)) for r in rgbs]))
    assert torch.equal(dep.cpu(), torch.stack([dep_tf(Image.fromarray(d).convert("L")) for d in deps]))


def test_batch_independence():
    pp = _pp()
    rgbs, deps = _batch(RAGGED, seed=3)
    img, dep = pp(rgbs, deps)
    for b in range(len(rgbs)):
        i1, d1 = pp(rgbs[b:b + 1], deps[b:b + 1])
        assert torch.equal(i1[0], img[b]) and torch.equal(d1[0], dep[b]), b


def test_large_photo():
    pp = _pp()
    g = np.random.default_rng(11)
    rgb, dep = _image(4000, 3000, 3, g), _image(3000, 4000, 3, g)
    got = pp([rgb], [dep])
    _check(got, _oracle([rgb], [dep], (384, 384)))


def test_b64_seeded_sizes():
    pp = _pp()
    g = np.random.default_rng(0)
    sizes = [(int(g.integers(250, 1501)), int(g.integers(250, 1501))) for _ in range(64)]
    rgbs, deps = _batch(sizes, seed=1)
    deps = [d if d.ndim == 3 else np.repeat(d[..., None], 3, 2) for d in deps]     # colour renderings throughout
    got = pp(rgbs, deps)
    _check(got, _oracle(rgbs, deps, (384, 384)))
    again = pp(rgbs, deps)                        # the staging buffer is reused; the result does not move
    assert torch.equal(again[0], got[0]) and torch.equal(again[1], got[1])


def test_custom_mean_std():
    pp = _pp()
    rgbs, deps = _batch([(600, 900), (300, 200), (384, 384)], seed=5)
    mean, std = (0.5, 0.25, 0.1), (0.3, 1.7, 0.05)
    got = pp(rgbs, deps, size=(352, 352), mean=mean, std=std)
    _check(got, _oracle(rgbs, deps, (352, 352), mean, std))
    T = pytest.importorskip("torchvision.transforms")
    Image = pytest.importorskip("PIL.Image")
    tf = T.Compose([T.Resize((352, 352)), T.ToTensor(), T.Normalize(mean, std)])
    assert torch.equal(got[0].cpu(), torch.stack([tf(Image.fromarray(r)) for r in rgbs]))


def test_rejects_bad_input():
    pp = _pp()
    rgb, dep = np.zeros((10, 12, 3), np.uint8), np.zeros((10, 12), np.uint8)
    bad = [
        ([], []),
        ([rgb, rgb], [dep]),
        ([rgb.astype(np.float32)], [dep]),
        ([rgb], [dep.astype(np.int16)]),
        ([torch.zeros(10, 12, 3)], [dep]),
        ([rgb[..., :2]], [dep]),
        ([rgb[..., 0]], [dep]),
        ([rgb], [np.zeros((10, 12, 2), np.uint8)]),
        ([np.zeros((0, 12, 3), np.uint8)], [dep]),
        ([rgb], [np.zeros((10, 0), np.uint8)]),
    ]
    for rgbs, deps in bad:
        with pytest.raises(ValueError):
            pp(rgbs, deps)
    with pytest.raises(ValueError):
        pp([rgb], [dep], std=(0.2, 0.0, 0.2))
    with pytest.raises(ValueError):
        pp([rgb], [dep], size=(0, 384))
