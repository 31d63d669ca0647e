"""Byte container shared by the compressed-tile formats (`jpeg.JpegBatch`, `png.PngBatch`): n files back to back in
one host or device buffer plus n + 1 host byte offsets.  The subclass names the format the bytes are decoded as."""
from __future__ import annotations

import numpy as np


class EncodedBatch:
    """n encoded files back to back: tile i is data[offsets[i]:offsets[i + 1]].

    data: 1-D uint8 numpy array (host) or contiguous CUDA torch uint8 tensor (read in place on the GPU);
    offsets: n + 1 non-decreasing int64 byte offsets (host)."""

    def __init__(self, data, offsets):
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        if offsets.ndim != 1 or offsets.size < 1:
            raise ValueError("offsets must be a 1-D array of n + 1 byte offsets")
        if isinstance(data, (bytes, bytearray, memoryview)):
            data = np.frombuffer(data, np.uint8)
        if isinstance(data, np.ndarray):
            data = np.ascontiguousarray(data.reshape(-1), dtype=np.uint8)
        else:
            if str(getattr(data, "dtype", "")) != "torch.uint8" or data.dim() != 1 or not data.is_contiguous():
                raise TypeError("data must be a 1-D uint8 numpy array or a contiguous 1-D torch.uint8 tensor")
        size = int(data.shape[0])
        if offsets[0] < 0 or np.any(np.diff(offsets) < 0) or offsets[-1] > size:
            raise ValueError("offsets must be non-decreasing and lie within data")
        self.data = data
        self.offsets = offsets

    @classmethod
    def from_bytes(cls, items):
        """from a list of encoded files (bytes)"""
        items = [bytes(b) for b in items]
        offsets = np.zeros(len(items) + 1, np.int64)
        offsets[1:] = np.cumsum([len(b) for b in items])
        return cls(np.frombuffer(b"".join(items), np.uint8).copy(), offsets)

    def __len__(self) -> int:
        return int(self.offsets.size - 1)

    @property
    def nbytes(self) -> int:
        return int(self.offsets[-1] - self.offsets[0])

    @property
    def on_device(self) -> bool:
        return not isinstance(self.data, np.ndarray)

    def tile(self, i: int) -> bytes:
        a, b = int(self.offsets[i]), int(self.offsets[i + 1])
        chunk = self.data[a:b]
        return bytes(chunk.cpu().numpy()) if self.on_device else chunk.tobytes()

    def cuda(self, device: int | None = None):
        """the same batch (same class) with its bytes in device memory"""
        import torch
        return type(self)(torch.from_numpy(np.asarray(self.data)).cuda(device), self.offsets)
