"""oracle/preprocess_ref.py against PIL and torchvision, bit for bit: the bilinear resample, the pass order,
convert('L') and the whole dataset transform.  CPU only; skipped where PIL or torchvision is missing."""
import numpy as np
import pytest
import torch

from oracle import preprocess_ref as P

Image = pytest.importorskip("PIL.Image")
T = pytest.importorskip("torchvision.transforms")

# (H, W): down/down, up/up, mixed, one axis unchanged (at 384), 1 x N / N x 1 / 1 x 1, odd sizes, a 4000 x 3000 photo
SIZES = [(1024, 768), (768, 1024), (200, 300), (5, 7), (250, 1500), (1500, 250), (384, 1000), (1000, 384),
         (384, 200), (200, 384), (384, 384), (1, 50), (50, 1), (1, 1), (1, 1000), (1000, 1), (383, 385),
         (4000, 3000)]
# the pass-order rule of Pillow's Image.resize: vertical first iff H > 100 W and the output is shorter than H.
# (800, 8), (3000, 30): exactly 100 -> horizontal first; (801, 8), (1000, 8), (2500, 24), (1400, 13): vertical first;
# (250, 2), (380, 3): taller than 100 W but growing to 384 rows -> horizontal first
BOUNDARY = [(800, 8), (801, 8), (3000, 30), (3001, 30), (1000, 8), (2500, 24), (1400, 13), (250, 2), (380, 3)]


def _content(h, w, c, seed, smooth):
    g = np.random.default_rng(seed)
    if not smooth:
        return g.integers(0, 256, (h, w, c), dtype=np.uint8)
    y, x = np.mgrid[0:h, 0:w]
    base = 127.5 + 100 * np.sin(x[..., None] * (0.01 + 0.02 * np.arange(c)) + y[..., None] * 0.013)
    return np.clip(base + g.normal(0, 4, (h, w, c)), 0, 255).astype(np.uint8)


def _pil(a, out):
    return np.asarray(Image.fromarray(a if a.shape[-1] != 1 else a[..., 0]).resize((out[1], out[0]),
                                                                                   Image.BILINEAR))


@pytest.mark.parametrize("smooth", [False, True], ids=["random", "smooth"])
@pytest.mark.parametrize("hw", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_resize_equals_pil(hw, smooth):
    a = _content(*hw, 3, seed=hw[0] * 7 + hw[1], smooth=smooth)
    for out in ((384, 384), (352, 352), (768, 768), (384, 200)):
        assert np.array_equal(P.resize(a, *out), _pil(a, out)), out


@pytest.mark.parametrize("hw", BOUNDARY, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("out", [(384, 384), (352, 352), (768, 768)], ids=lambda s: f"{s[0]}")
def test_pass_order_boundary(hw, out):
    a = _content(*hw, 1, seed=hw[0] + hw[1], smooth=False)[..., 0]
    ref = _pil(a[..., None], out)
    assert np.array_equal(P.resize(a, *out), ref)
    vf = P.vertical_first(hw[0], hw[1], out[0])
    assert vf == (hw[0] > 100 * hw[1] and out[0] < hw[0])
    # the other order gives other bits on these sizes: the rule is what makes the oracle match
    assert not np.array_equal(P.resize(a, *out, order="h" if vf else "v"), ref)


def test_rule_needs_the_shrink_condition():
    """A source more than 100 times taller than wide that grows is resized horizontally first; a rule on the aspect
    ratio alone would pick the vertical pass and miss."""
    a = _content(250, 2, 3, seed=5, smooth=False)
    ref = _pil(a, (384, 384))
    assert np.array_equal(P.resize(a, 384, 384, order="h"), ref)
    assert not np.array_equal(P.resize(a, 384, 384, order="v"), ref)


def test_float_resample_fails():
    """A one-pass float resample (same weights, no uint8 intermediate) misses PIL's bits: the two-pass integer
    arithmetic is needed."""
    a = _content(1024, 768, 3, seed=1, smooth=True)
    xmin, n, kx = P.coeffs(768, 384)
    ymin, m, ky = P.coeffs(1024, 384)

    def mat(lo, cnt, k, size):
        M = np.zeros((len(lo), size))
        for o in range(len(lo)):
            M[o, lo[o]:lo[o] + cnt[o]] = k[o, :cnt[o]] / float(1 << P.PRECISION_BITS)
        return M

    Wy, Wx = mat(ymin, m, ky, 1024), mat(xmin, n, kx, 768)
    rows = np.tensordot(Wy, a.astype(np.float64), axes=(1, 0))                    # (384, 768, 3)
    flt = np.clip(np.rint(np.tensordot(rows, Wx, axes=(1, 1)).transpose(0, 2, 1)), 0, 255).astype(np.uint8)
    ref = _pil(a, (384, 384))
    assert np.array_equal(P.resize(a, 384, 384), ref)
    assert (flt != ref).sum() > 1000


def test_luma_equals_convert_l():
    r, g = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")          # every (R, G) pair, B descending
    a = np.stack([r, g, 255 - r], -1).astype(np.uint8)
    a = np.concatenate([a, _content(300, 256, 3, seed=2, smooth=False)])
    assert np.array_equal(P.to_luma(a), np.asarray(Image.fromarray(a).convert("L")))


@pytest.mark.parametrize("size", [(384, 384), (352, 352), (200, 500)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_whole_transform_equals_torchvision(size):
    mean, std = P.IMAGENET_MEAN, P.IMAGENET_STD
    rgb_tf = T.Compose([T.Resize(size), T.ToTensor(), T.Normalize(mean, std)])
    dep_tf = T.Compose([T.Resize(size), T.ToTensor()])
    for k, (hw, dhw) in enumerate([((1024, 768), (1024, 768)), ((600, 900), (300, 450)), ((1000, 8), (5, 7))]):
        rgb = _content(*hw, 3, seed=k, smooth=True)
        for dep in (_content(*dhw, 3, seed=k + 10, smooth=True), _content(*dhw, 1, seed=k + 20, smooth=False)[..., 0]):
            want_rgb = rgb_tf(Image.fromarray(rgb)).numpy()
            want_dep = dep_tf(Image.fromarray(dep).convert("L")).numpy()
            assert np.array_equal(P.preprocess_rgb(rgb, size), want_rgb)
            assert np.array_equal(P.preprocess_depth(dep, size), want_dep)
    # every lookup entry, for the ImageNet and for other mean / std
    u = np.arange(256, dtype=np.uint8)[None, :, None].repeat(3, 2)
    for m, s in ((mean, std), ((0.5, 0.25, 0.1), (0.3, 1.7, 0.05))):
        got = P.lut(m, s)
        want = T.Normalize(m, s)(T.ToTensor()(Image.fromarray(u))).numpy()[:, 0]
        assert np.array_equal(got, want)
    assert np.array_equal(P.lut()[0], T.ToTensor()(Image.fromarray(u[..., 0])).numpy()[0, 0])
    assert torch.equal(torch.from_numpy(P.lut()[0]), torch.arange(256, dtype=torch.float32) / 255)
