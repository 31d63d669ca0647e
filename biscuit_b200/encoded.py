"""Compressed tiles of any format (`jpeg.JpegBatch`, `png.PngBatch`): the byte container -- n files back to back in one
host or device buffer plus n + 1 host byte offsets -- and the calls into the library's `bq_{fmt}_*` entry points that
`jpeg` and `png` expose.  The subclass names the format the bytes are decoded as (`FORMAT`)."""
from __future__ import annotations

import numpy as np

from . import _ffi


class EncodedBatch:
    """n encoded files back to back: tile i is data[offsets[i]:offsets[i + 1]].

    data: 1-D uint8 numpy array (host) or contiguous CUDA torch uint8 tensor (read in place on the GPU);
    offsets: n + 1 non-decreasing int64 byte offsets (host)."""

    FORMAT: str          # "jpeg" / "png": the `bq_{FORMAT}_*` entry points that decode it
    # decode options as the `flags` of the `bq_{FORMAT}_*_ex` entry points; None: the format has none
    flags: int | None = None
    # whether the header parse depends on those options, so that inspect takes them too (`bq_{FORMAT}_inspect_ex`)
    PARSE_OPTIONS = False

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
    def from_bytes(cls, items, **options):
        """from a list of encoded files (bytes); `options` are the subclass's decode options"""
        items = [bytes(b) for b in items]
        offsets = np.zeros(len(items) + 1, np.int64)
        offsets[1:] = np.cumsum([len(b) for b in items])
        return cls(np.frombuffer(b"".join(items), np.uint8).copy(), offsets, **options)

    def options(self) -> dict:
        """the constructor's decode-option arguments of this batch"""
        return {}

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
        """the same batch (same class, same decode options) with its bytes in device memory"""
        import torch
        return type(self)(torch.from_numpy(np.asarray(self.data)).cuda(device), self.offsets, **self.options())


def status_message(fmt: str, code: int) -> str:
    return getattr(_ffi.load_library(), f"bq_{fmt}_status_string")(int(code)).decode()


def inspect(fmt: str, batch: EncodedBatch, px: int) -> np.ndarray:
    if batch.on_device:
        raise ValueError("inspect reads host bytes; the batch is in device memory")
    name, flags = entry_point(f"bq_{fmt}_inspect", batch) if batch.PARSE_OPTIONS else (f"bq_{fmt}_inspect", ())
    st = np.zeros(len(batch), np.int32)
    rc = getattr(_ffi.load_library(), name)(_ffi.ptr(batch.data), _ffi.ptr(batch.offsets), len(batch), int(px), *flags,
                                             _ffi.ptr(st))
    if rc != 0:
        raise ValueError(f"{name}: bad argument")
    return st


def check(fmt: str, batch: EncodedBatch, px: int) -> None:
    st = inspect(fmt, batch, px)
    bad = np.flatnonzero(st)
    if bad.size:
        raise ValueError(f"{fmt.upper()} tile {int(bad[0])}: {status_message(fmt, int(st[bad[0]]))}")


def decode(fmt: str, batch: EncodedBatch, px: int, ctx: _ffi.Context | None, out):
    ctx = ctx or _ffi.default_context()
    n = len(batch)
    if out is None:
        out = np.empty((n, px, px, 3), np.uint8)
    if tuple(out.shape) != (n, px, px, 3) or str(out.dtype).replace("torch.", "") != "uint8":
        raise ValueError(f"out must be uint8 of shape {(n, px, px, 3)}")
    if isinstance(out, np.ndarray) and not out.flags.c_contiguous:
        raise ValueError("out must be C-contiguous")
    st = np.zeros(n, np.int32)
    name, flags = entry_point(f"bq_{fmt}_decode", batch)
    _ffi.check(ctx.handle, getattr(ctx.lib, name)(ctx.handle, _ffi.ptr(batch.data), _ffi.ptr(batch.offsets), n, int(px),
                                                  *flags, _ffi.ptr(out), _ffi.ptr(st)), name)
    return out


def entry_point(name: str, batch: EncodedBatch):
    """(entry point, extra arguments) that decode `batch` with its options: `name` itself, or `name`_ex and its
    flags argument"""
    return (name, ()) if batch.flags is None else (name + "_ex", (int(batch.flags),))
