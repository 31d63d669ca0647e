"""JPEG tiles decoded on the GPU (csrc/jpeg.cu, csrc/jpeg_sm100.cuh).

A `JpegBatch` holds n JPEG files back to back.  `decode(batch)` returns the uint8 tiles, byte for byte what
`np.asarray(PIL.Image.open(io.BytesIO(b)).convert("RGB"))` gives (libjpeg-turbo's default decode: JDCT_ISLOW IDCT,
fancy upsampling, jdcolor.c YCbCr->RGB), and `UncertaintyInterface.predict(batch)` runs MC-dropout inference on them
with the decode in front of the backbone, micro-batch by micro-batch.

The batch also carries the two decode options of TensorFlow's `tf.image.decode_jpeg`, under its names:
`dct_method="INTEGER_FAST"` (or `""`, which TensorFlow maps to it) selects libjpeg-turbo's JDCT_IFAST IDCT, and
`fancy_upscaling=False` replicates 4:2:2 / 4:2:0 chroma instead of interpolating it.  `decode_jpeg` with its defaults
decodes with INTEGER_FAST and fancy upscaling (per TensorFlow's decode_image_op.cc), so that pair is the decode to pick
for models trained on tiles TensorFlow decoded.  With both options the tiles equal libjpeg-turbo's IFAST decode without
fancy upsampling byte for byte (the decoder TensorFlow links); equality with TensorFlow's own output is not verified.

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


# tf.image.decode_jpeg's dct_method values -> IDCT flag; like TensorFlow, "" means INTEGER_FAST
DCT_METHODS = {"INTEGER_ACCURATE": 0, "INTEGER_FAST": _ffi.BQ_JPEG_IDCT_IFAST, "": _ffi.BQ_JPEG_IDCT_IFAST}


def check_dct_method(dct_method) -> None:
    if not isinstance(dct_method, str) or dct_method not in DCT_METHODS:
        raise ValueError(f"dct_method must be 'INTEGER_ACCURATE', 'INTEGER_FAST' or '' (INTEGER_FAST), "
                         f"got {dct_method!r}")


class JpegBatch(EncodedBatch):
    """n JPEG files back to back: tile i is data[offsets[i]:offsets[i + 1]].

    data: 1-D uint8 numpy array (host) or contiguous CUDA torch uint8 tensor (read in place on the GPU);
    offsets: n + 1 non-decreasing int64 byte offsets (host).
    dct_method, fancy_upscaling: how the tiles are decoded, as in `tf.image.decode_jpeg` (module docstring); the
    defaults are libjpeg-turbo's default decode."""

    FORMAT = "jpeg"

    def __init__(self, data, offsets, dct_method: str = "INTEGER_ACCURATE", fancy_upscaling: bool = True):
        check_dct_method(dct_method)
        if not isinstance(fancy_upscaling, (bool, np.bool_)):
            raise ValueError(f"fancy_upscaling must be a bool, got {fancy_upscaling!r}")
        super().__init__(data, offsets)
        self.dct_method = dct_method
        self.fancy_upscaling = bool(fancy_upscaling)

    @property
    def flags(self) -> int:
        return DCT_METHODS[self.dct_method] | (0 if self.fancy_upscaling else _ffi.BQ_JPEG_REPLICATE_CHROMA)

    def options(self) -> dict:
        return dict(dct_method=self.dct_method, fancy_upscaling=self.fancy_upscaling)


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
    """uint8 NHWC [n, px, px, 3] tiles decoded on the GPU with the batch's decode options.  `out` may be a preallocated
    numpy array or CUDA torch tensor of that shape (device output stays on the device); default: a new numpy array."""
    return encoded.decode("jpeg", batch, px, ctx, out)


def last_stats(ctx: _ffi.Context | None = None) -> dict:
    """subsequence statistics of the last `decode` on ctx"""
    ctx = ctx or _ffi.default_context()
    s = (C.c_int64 * 4)()
    _ffi.check(ctx.handle, ctx.lib.bq_jpeg_last_stats(ctx.handle, s), "bq_jpeg_last_stats")
    return dict(tiles=int(s[0]), subsequences=int(s[1]), max_sync_rounds=int(s[2]), redecoded=int(s[3]))
