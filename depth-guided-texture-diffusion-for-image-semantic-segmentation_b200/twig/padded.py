"""A batch of single-channel maps of different sizes, as the public COD test sets give their ground truths.

Image b occupies the top-left H_b x W_b of plane b of one (B, 1, Hmax, Wmax) fp32 buffer.  The rest of each plane is
undefined and no kernel reads it.  The kernels take the sizes as a device (B, 2) int32 array, which is built here from
sizes the host already knows, checked here, and uploaded once with a pinned, non-blocking copy.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch

__all__ = ["PaddedBatch"]


class PaddedBatch:
    """`data` (B, 1, Hmax, Wmax) fp32 and `sizes`, B pairs (H_b, W_b) with 2 <= H_b <= Hmax and 2 <= W_b <= Wmax."""

    def __init__(self, data: torch.Tensor, sizes: Sequence[Tuple[int, int]]):
        if data.dim() != 4 or data.shape[1] != 1:
            raise ValueError(f"PaddedBatch: data must be (B, 1, Hmax, Wmax), got {tuple(data.shape)}")
        B, _, Hmax, Wmax = data.shape
        sizes = tuple((int(h), int(w)) for h, w in sizes)
        if len(sizes) != B:
            raise ValueError(f"PaddedBatch: {len(sizes)} sizes for {B} images")
        for b, (h, w) in enumerate(sizes):
            if not (2 <= h <= Hmax and 2 <= w <= Wmax):
                raise ValueError(f"PaddedBatch: image {b} is {h} x {w}; each side must be at least 2 and fit the "
                                 f"{Hmax} x {Wmax} buffer")
        self.data = data
        self.sizes = sizes
        self._device_sizes: Optional[torch.Tensor] = None

    @classmethod
    def from_list(cls, maps: Sequence[torch.Tensor], device: Optional[torch.device] = None) -> "PaddedBatch":
        """Pack per-image (1, H, W) or (H, W) maps, one slice copy each, into a new fp32 buffer on `device` (default:
        the device of the first map)."""
        if len(maps) == 0:
            raise ValueError("PaddedBatch.from_list: no maps")
        for m in maps:
            if not (m.dim() == 2 or (m.dim() == 3 and m.shape[0] == 1)):
                raise ValueError(f"PaddedBatch.from_list: maps must be (1, H, W) or (H, W), got {tuple(m.shape)}")
        sizes = [(int(m.shape[-2]), int(m.shape[-1])) for m in maps]
        Hmax, Wmax = max(h for h, _ in sizes), max(w for _, w in sizes)
        data = torch.empty(len(maps), 1, Hmax, Wmax, device=device or maps[0].device, dtype=torch.float32)
        batch = cls(data, sizes)
        with torch.no_grad():
            for b, ((h, w), m) in enumerate(zip(sizes, maps)):
                data[b, 0, :h, :w].copy_(m.reshape(h, w), non_blocking=True)
        return batch

    def empty_like(self) -> "PaddedBatch":
        """A new, uninitialised buffer with the same sizes (and the same uploaded device sizes)."""
        out = PaddedBatch(torch.empty_like(self.data), self.sizes)
        out._device_sizes = self._device_sizes
        return out

    def device_sizes(self) -> torch.Tensor:
        """The sizes as a (B, 2) int32 tensor on the buffer's device, uploaded on first use."""
        if self._device_sizes is None:
            host = torch.tensor(self.sizes, dtype=torch.int32)
            if self.data.is_cuda:
                host = host.pin_memory()
            self._device_sizes = host.to(self.data.device, non_blocking=True)
        return self._device_sizes

    def unbind(self) -> List[torch.Tensor]:
        """Per-image (1, H_b, W_b) views of the buffer."""
        return [self.data[b, :, :h, :w] for b, (h, w) in enumerate(self.sizes)]

    def __len__(self) -> int:
        return len(self.sizes)
