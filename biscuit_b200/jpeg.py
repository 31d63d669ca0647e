"""JPEG tiles decoded on the GPU (csrc/jpeg.cu, csrc/jpeg_sm100.cuh).

A `JpegBatch` holds n JPEG files back to back.  `decode(batch)` returns the uint8 tiles, byte for byte what
`np.asarray(PIL.Image.open(io.BytesIO(b)).convert("RGB"))` gives (libjpeg-turbo's default decode: JDCT_ISLOW IDCT,
fancy upsampling, jdcolor.c YCbCr->RGB), and `UncertaintyInterface.predict(batch)` runs MC-dropout inference on them
with the decode in front of the backbone, micro-batch by micro-batch.

Accepted: baseline / extended sequential Huffman JPEG, 8-bit, 3 components (YCbCr), sampling 4:4:4, 4:2:2 or 4:2:0,
any quantisation / Huffman tables, restart intervals, APPn / COM segments, size tile_px x tile_px.  Everything else
raises ValueError naming the tile before anything runs on the GPU; an entropy-coded segment that is truncated or holds
an invalid code raises ValueError naming the tile after the batch.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _ffi, encoded
from .encoded import EncodedBatch
from .hp import nature2022


class JpegBatch(EncodedBatch):
    """n JPEG files back to back: tile i is data[offsets[i]:offsets[i + 1]].

    data: 1-D uint8 numpy array (host) or contiguous CUDA torch uint8 tensor (read in place on the GPU);
    offsets: n + 1 non-decreasing int64 byte offsets (host)."""

    FORMAT = "jpeg"


def status_message(code: int) -> str:
    return encoded.status_message("jpeg", code)


def inspect(batch: JpegBatch, px: int = nature2022.tile_px) -> np.ndarray:
    """Host marker parse of every tile, no GPU needed: int32 status per tile (0 = accepted, else a BQ_JPEG_* code,
    see `status_message`)."""
    return encoded.inspect("jpeg", batch, px)


def check(batch: JpegBatch, px: int = nature2022.tile_px) -> None:
    """raise ValueError for the first tile `decode` would reject by its headers"""
    return encoded.check("jpeg", batch, px)


def decode(batch: JpegBatch, px: int = nature2022.tile_px, ctx: _ffi.Context | None = None, out=None):
    """uint8 NHWC [n, px, px, 3] tiles decoded on the GPU.  `out` may be a preallocated numpy array or CUDA torch tensor
    of that shape (device output stays on the device); default: a new numpy array."""
    return encoded.decode("jpeg", batch, px, ctx, out)


def last_stats(ctx: _ffi.Context | None = None) -> dict:
    """subsequence statistics of the last `decode` on ctx"""
    ctx = ctx or _ffi.default_context()
    s = (C.c_int64 * 4)()
    _ffi.check(ctx.handle, ctx.lib.bq_jpeg_last_stats(ctx.handle, s), "bq_jpeg_last_stats")
    return dict(tiles=int(s[0]), subsequences=int(s[1]), max_sync_rounds=int(s[2]), redecoded=int(s[3]))
