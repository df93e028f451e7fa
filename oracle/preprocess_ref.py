"""CPU restatement of the datasets' host transforms for one RGB-D pair (SURVEY §2 row 11): PIL 12.2's bilinear
`Image.resize` of an 8-bit image, `convert('L')`, torchvision's `ToTensor` and ImageNet `Normalize`.

TEST INFRASTRUCTURE ONLY: imported by tests/ and tools/; never by the product path.

Plain numpy, on purpose without PIL or torchvision, so that the GPU tests run where those are absent.
tests/test_oracle_preprocess.py checks every function here against PIL and torchvision bit for bit.

The resample (Pillow `src/libImaging/Resample.c`, `precompute_coeffs`, `normalize_coeffs_8bpc`,
`ImagingResampleHorizontal_8bpc` / `Vertical_8bpc`):
  - per axis, float64 coefficients of the triangle filter widened by the downscale factor, normalised to sum 1,
    then rounded to int32 with 22 fraction bits;
  - each pass accumulates u8 * k in int32 from 2^21 and keeps clip8(acc >> 22): the intermediate between the two
    passes is uint8, so no one-pass float resample reproduces it;
  - an axis whose size does not change is skipped;
  - the horizontal pass runs first, except when the source is more than 100 times taller than wide AND the output
    is shorter than the source: then the vertical pass runs first (the branch in Pillow's `Image.resize`).
"""
from __future__ import annotations

import math
from typing import Sequence, Tuple

import numpy as np

PRECISION_BITS = 22          # 32 - 8 - 2
IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


def coeffs(in_size: int, out_size: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """-> (xmin (out,), n (out,), k (out, ksize) int64): output index i reads source [xmin, xmin + n) with the
    fixed-point weights k[i, :n] (0 beyond n).  Float64 in PIL's operation order; Python floats are IEEE doubles
    and nothing is contracted into an FMA."""
    scale = float(in_size) / out_size
    fs = max(scale, 1.0)
    support = 1.0 * fs                        # bilinear support is 1
    ksize = int(math.ceil(support)) * 2 + 1
    ss = 1.0 / fs
    xmin_a = np.zeros(out_size, np.int64)
    n_a = np.zeros(out_size, np.int64)
    kk = np.zeros((out_size, ksize), np.int64)
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        ws = []
        for x in range(xmax):
            t = abs((x + xmin - center + 0.5) * ss)
            ws.append(1.0 - t if t < 1.0 else 0.0)
        ww = sum_seq(ws)
        for x, w in enumerate(ws):
            if ww != 0.0:
                w = w / ww
            kk[xx, x] = int(0.5 + w * (1 << PRECISION_BITS))
        xmin_a[xx], n_a[xx] = xmin, xmax
    return xmin_a, n_a, kk


def sum_seq(ws: Sequence[float]) -> float:
    """Left-to-right float64 sum (PIL's `ww += w`)."""
    s = 0.0
    for w in ws:
        s += w
    return s


def resample_axis1(img: np.ndarray, out_size: int) -> np.ndarray:
    """One pass along axis 1 of an (H, W, C) uint8 array -> (H, out_size, C) uint8."""
    xmin, n, kk = coeffs(img.shape[1], out_size)
    acc = np.full((img.shape[0], out_size, img.shape[2]), 1 << (PRECISION_BITS - 1), np.int64)
    for i in range(kk.shape[1]):
        idx = np.minimum(xmin + i, img.shape[1] - 1)                  # taps past n carry k = 0
        acc += img[:, idx, :].astype(np.int64) * np.where(i < n, kk[:, i], 0)[None, :, None]
    return np.clip(acc >> PRECISION_BITS, 0, 255).astype(np.uint8)


def horizontal(img: np.ndarray, out_w: int) -> np.ndarray:
    return resample_axis1(img, out_w)


def vertical(img: np.ndarray, out_h: int) -> np.ndarray:
    return resample_axis1(img.transpose(1, 0, 2), out_h).transpose(1, 0, 2)


def vertical_first(h: int, w: int, out_h: int) -> bool:
    """Pillow's pass order: vertical first for a source more than 100 times taller than wide that gets shorter."""
    return h > 100 * w and out_h < h


def resize(img: np.ndarray, out_h: int, out_w: int, order: str = "pil") -> np.ndarray:
    """`Image.resize((out_w, out_h), BILINEAR)` of an (H, W) or (H, W, C) uint8 array.  order = "pil" (the rule
    above), "h" or "v" (forced: for the tests that show the rule matters)."""
    a = img[..., None] if img.ndim == 2 else img
    H, W = a.shape[:2]
    vfirst = vertical_first(H, W, out_h) if order == "pil" else order == "v"
    h = (lambda x: horizontal(x, out_w)) if W != out_w else (lambda x: x)
    v = (lambda x: vertical(x, out_h)) if H != out_h else (lambda x: x)
    out = h(v(a)) if vfirst else v(h(a))
    return np.ascontiguousarray(out[..., 0] if img.ndim == 2 else out)


def to_luma(rgb: np.ndarray) -> np.ndarray:
    """`convert('L')` of an (H, W, 3) uint8 array (ITU-R 601-2 in 16-bit fixed point)."""
    r, g, b = (rgb[..., c].astype(np.int64) for c in range(3))
    return ((19595 * r + 38470 * g + 7471 * b + 0x8000) >> 16).astype(np.uint8)


def lut(mean: Sequence[float] = None, std: Sequence[float] = None) -> np.ndarray:
    """(C, 256) float32: `ToTensor` (u / 255) and, with mean / std, `Normalize` ((x - mean) / std), each a correctly
    rounded fp32 operation as torch runs them on the host."""
    u = np.arange(256, dtype=np.float32) / np.float32(255)
    if mean is None:
        return u[None]
    m = np.asarray(mean, np.float32)[:, None]
    s = np.asarray(std, np.float32)[:, None]
    return ((u[None] - m) / s).astype(np.float32)


def preprocess_rgb(rgb: np.ndarray, size: Tuple[int, int], mean=IMAGENET_MEAN, std=IMAGENET_STD) -> np.ndarray:
    """`Compose([Resize(size), ToTensor(), Normalize(mean, std)])(Image.fromarray(rgb))` -> (3, S_h, S_w) float32."""
    u8 = resize(rgb, size[0], size[1])
    t = lut(mean, std)
    return np.stack([t[c][u8[..., c]] for c in range(3)])


def preprocess_depth(depth: np.ndarray, size: Tuple[int, int]) -> np.ndarray:
    """`Compose([Resize(size), ToTensor()])(Image.fromarray(depth).convert('L'))` -> (1, S_h, S_w) float32, for an
    (H, W) or (H, W, 3) uint8 array."""
    gray = to_luma(depth) if depth.ndim == 3 else depth
    return lut()[0][resize(gray, size[0], size[1])][None]
