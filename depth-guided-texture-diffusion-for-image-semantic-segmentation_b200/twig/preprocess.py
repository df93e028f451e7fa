"""Decoded RGB-D images of any size -> the model's input tensors, on the GPU (csrc/preprocess_ops.cu).

The reference datasets (SURVEY §2 row 11, e.g. `twig/dataset/sod_train.py`) transform each image on the host:
`Resize((384, 384))`, `ToTensor`, ImageNet `Normalize` for the RGB, and for the depth, opened as 'L', `convert('L')`,
`Resize`, `ToTensor`.  `preprocess_rgbd` returns, bit for bit, what those transforms give, for a whole batch of
images of different sizes in four kernel launches.

The host packs every plane, with a descriptor table at its head, into one pinned uint8 staging buffer that is reused
across calls, and copies it to the device with one non-blocking copy.  No call waits for the device except when the
staging buffer is about to be overwritten while the previous call's copy is still in flight.
"""
from __future__ import annotations

import threading
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .ops import capi
from .ops.capi import call, ptr

__all__ = ["preprocess_rgbd", "IMAGENET_MEAN", "IMAGENET_STD"]

IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)
DESC_FIELDS = 7          # RGB offset, H, W, depth offset, H', W', depth channels
MAX_SIDE = 65535


def _as_u8(a, what: str, b: int) -> np.ndarray:
    if isinstance(a, torch.Tensor):
        if a.device.type != "cpu":
            raise ValueError(f"preprocess_rgbd: {what} {b} is on {a.device}; decoded images are host arrays")
        if a.dtype != torch.uint8:
            raise ValueError(f"preprocess_rgbd: {what} {b} has dtype {a.dtype}, expected uint8")
        return a.numpy()
    a = np.asarray(a)
    if a.dtype != np.uint8:
        raise ValueError(f"preprocess_rgbd: {what} {b} has dtype {a.dtype}, expected uint8")
    return a


def _check(rgbs, depths) -> Tuple[List[np.ndarray], List[np.ndarray]]:
    if len(rgbs) == 0:
        raise ValueError("preprocess_rgbd: no images")
    if len(rgbs) != len(depths):
        raise ValueError(f"preprocess_rgbd: {len(rgbs)} RGB images and {len(depths)} depth maps")
    if len(rgbs) > 65535:
        raise ValueError(f"preprocess_rgbd: at most 65535 images per call, got {len(rgbs)}")
    rs, ds = [], []
    for b, (r, d) in enumerate(zip(rgbs, depths)):
        r, d = _as_u8(r, "RGB image", b), _as_u8(d, "depth map", b)
        if r.ndim != 3 or r.shape[2] != 3:
            raise ValueError(f"preprocess_rgbd: RGB image {b} has shape {r.shape}, expected (H, W, 3)")
        if not (d.ndim == 2 or (d.ndim == 3 and d.shape[2] == 3)):
            raise ValueError(f"preprocess_rgbd: depth map {b} has shape {d.shape}, expected (H, W) or (H, W, 3)")
        for name, a in (("RGB image", r), ("depth map", d)):
            if not (1 <= a.shape[0] <= MAX_SIDE and 1 <= a.shape[1] <= MAX_SIDE):
                raise ValueError(f"preprocess_rgbd: {name} {b} is {a.shape[0]} x {a.shape[1]}; each side must be "
                                 f"1 to {MAX_SIDE}")
        rs.append(r)
        ds.append(d)
    return rs, ds


class _Staging:
    """One growing pinned buffer per device.  `event` records the end of the last copy out of it; the buffer is
    rewritten only after that event has completed."""

    def __init__(self):
        self.buf: Optional[torch.Tensor] = None
        self.event: Optional[torch.cuda.Event] = None

    def acquire(self, nbytes: int) -> torch.Tensor:
        if self.event is not None:
            self.event.synchronize()
        if self.buf is None or self.buf.numel() < nbytes:
            # freeing the old buffer is safe: torch's pinned-memory allocator holds a block until the copies that
            # read it have finished
            self.buf = torch.empty(max(nbytes, 1 << 20) * 5 // 4, dtype=torch.uint8, pin_memory=True)
        return self.buf


_staging = {}
_lock = threading.Lock()


def preprocess_rgbd(rgbs: Sequence, depths: Sequence, size: Tuple[int, int] = (384, 384),
                    mean: Sequence[float] = IMAGENET_MEAN, std: Sequence[float] = IMAGENET_STD,
                    device="cuda") -> Tuple[torch.Tensor, torch.Tensor]:
    """rgbs: B uint8 (H_b, W_b, 3) arrays (numpy, e.g. `np.asarray(pil_image)`, or CPU tensors); depths: B uint8
    (H'_b, W'_b) or (H'_b, W'_b, 3) arrays, three channels being converted with PIL's 'L' formula.  Sizes may differ
    from image to image and between an image's RGB and depth.

    -> image (B, 3, S_h, S_w) and depth (B, 1, S_h, S_w) fp32, contiguous, on `device`, equal bit for bit to
    `T.Compose([T.Resize(size), T.ToTensor(), T.Normalize(mean, std)])(Image.fromarray(rgb))` and to
    `T.Compose([T.Resize(size), T.ToTensor()])(Image.fromarray(d).convert('L'))`, stacked.

    Raises ValueError, before anything is copied, for empty or unequal lists, a dtype other than uint8, a wrong
    channel count, a side of 0, a bad size or a zero std.  The results are ready in stream order on the current
    stream; the call does not wait for them."""
    rs, ds = _check(rgbs, depths)
    S_h, S_w = (int(v) for v in size)
    if not (1 <= S_h <= MAX_SIDE and 1 <= S_w <= MAX_SIDE):
        raise ValueError(f"preprocess_rgbd: bad output size {size}")
    mean32, std32 = np.asarray(mean, np.float32), np.asarray(std, np.float32)
    if mean32.shape != (3,) or std32.shape != (3,):
        raise ValueError("preprocess_rgbd: mean and std take three values")
    if (std32 == 0).any():
        raise ValueError(f"preprocess_rgbd: std evaluated to zero: {tuple(std)}")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError(f"preprocess_rgbd: runs on a CUDA device, got {dev}")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())

    with _lock, torch.cuda.device(dev):
        desc, total = _layout(rs, ds)
        st = _staging.setdefault(dev.index, _Staging())
        host = st.acquire(total)
        _fill(host.numpy(), desc, rs, ds)
        packed = torch.empty(total, dtype=torch.uint8, device=dev)
        packed.copy_(host[:total], non_blocking=True)
        if st.event is None:
            st.event = torch.cuda.Event()
        st.event.record()
        return _launch(packed, host, desc, (S_h, S_w), mean32, std32)


def _layout(rs: Sequence[np.ndarray], ds: Sequence[np.ndarray]) -> Tuple[np.ndarray, int]:
    """-> (descriptor table (B, 7) int64, packed bytes): the table at the head, then each image's RGB and depth."""
    B = len(rs)
    desc = np.zeros((B, DESC_FIELDS), np.int64)
    off = B * DESC_FIELDS * 8
    for b, (r, d) in enumerate(zip(rs, ds)):
        desc[b, 0:3] = off, r.shape[0], r.shape[1]
        off += r.size
        desc[b, 3:7] = off, d.shape[0], d.shape[1], 1 if d.ndim == 2 else 3
        off += d.size
    return desc, off


def _fill(view: np.ndarray, desc: np.ndarray, rs: Sequence[np.ndarray], ds: Sequence[np.ndarray]) -> None:
    """Write the table and every plane into the host byte buffer `view`."""
    view[:desc.size * 8] = desc.reshape(-1).view(np.uint8)
    for b, (r, d) in enumerate(zip(rs, ds)):
        view[desc[b, 0]:desc[b, 0] + r.size].reshape(r.shape)[...] = r
        view[desc[b, 3]:desc[b, 3] + d.size].reshape(d.shape)[...] = d


def _launch(packed: torch.Tensor, host: torch.Tensor, desc: np.ndarray, size: Tuple[int, int], mean32: np.ndarray,
            std32: np.ndarray) -> Tuple[torch.Tensor, torch.Tensor]:
    """The four launches on the current stream, from the device copy `packed` of the host buffer `host` (whose head
    the library reads to size the workspace)."""
    B, dev = len(desc), packed.device
    S_h, S_w = size
    ws_bytes = int(capi.load().dgtd_rgbd_preprocess_ws_bytes(host.data_ptr(), B, S_h, S_w))
    if ws_bytes < 0:
        raise RuntimeError(f"dgtd_rgbd_preprocess_ws_bytes failed: {capi.last_error()}")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    image = torch.empty(B, 3, S_h, S_w, dtype=torch.float32, device=dev)
    depth = torch.empty(B, 1, S_h, S_w, dtype=torch.float32, device=dev)
    max_h = int(max(desc[:, 1].max(), desc[:, 4].max()))
    max_w = int(max(desc[:, 2].max(), desc[:, 5].max()))
    call("dgtd_rgbd_preprocess_fwd", ptr(packed), packed.numel(), B, max_h, max_w, S_h, S_w,
         *(float(v) for v in mean32), *(float(v) for v in std32), ptr(ws), ws_bytes, ptr(image), ptr(depth),
         torch.cuda.current_stream(dev).cuda_stream)
    return image, depth
