"""PNG tiles decoded on the GPU (csrc/png.cu, csrc/png_sm100.cuh).

A `PngBatch` holds n PNG files back to back.  `decode(batch)` returns the uint8 tiles, byte for byte what
`np.asarray(PIL.Image.open(io.BytesIO(b)).convert("RGB"))` gives (PNG is lossless: these are the encoded pixels, and
also what TensorFlow's `decode_png` returns), and `UncertaintyInterface.predict(batch)` runs MC-dropout inference on
them with the decode in front of the backbone, micro-batch by micro-batch.

Accepted: 8-bit RGB (colour type 2), non-interlaced, size tile_px x tile_px, any zlib level / strategy / window size,
IDAT split into chunks of any size, ancillary chunks and PLTE anywhere (skipped).  Every other header raises
ValueError naming the tile before anything runs on the GPU; a DEFLATE stream, Adler-32 or filter byte that is corrupt
raises ValueError naming the tile after the batch.  Stricter than Pillow on corrupt data: a missing Adler-32 and a
stream that decompresses to more bytes than the image are rejected.
"""
from __future__ import annotations

import numpy as np

from . import _ffi, encoded
from .encoded import EncodedBatch
from .hp import nature2022

SIGNATURE = b"\x89PNG\r\n\x1a\n"


class PngBatch(EncodedBatch):
    """n PNG files back to back: tile i is data[offsets[i]:offsets[i + 1]].

    data: 1-D uint8 numpy array (host) or contiguous CUDA torch uint8 tensor (read in place on the GPU);
    offsets: n + 1 non-decreasing int64 byte offsets (host)."""

    FORMAT = "png"


def status_message(code: int) -> str:
    return encoded.status_message("png", code)


def inspect(batch: PngBatch, px: int = nature2022.tile_px) -> np.ndarray:
    """Host chunk parse of every tile, no GPU needed: int32 status per tile (0 = accepted, else a BQ_PNG_* code, see
    `status_message`)."""
    return encoded.inspect("png", batch, px)


def check(batch: PngBatch, px: int = nature2022.tile_px) -> None:
    """raise ValueError for the first tile `decode` would reject by its headers"""
    return encoded.check("png", batch, px)


def decode(batch: PngBatch, px: int = nature2022.tile_px, ctx: _ffi.Context | None = None, out=None):
    """uint8 NHWC [n, px, px, 3] tiles decoded on the GPU.  `out` may be a preallocated numpy array or CUDA torch tensor
    of that shape (device output stays on the device); default: a new numpy array."""
    return encoded.decode("png", batch, px, ctx, out)
