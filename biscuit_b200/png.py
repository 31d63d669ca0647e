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

With `convert_rgb=True` the batch decodes every PNG the specification allows, as TensorFlow's
`decode_png(channels=3)` and Pillow's `convert("RGB")` do: grayscale (1, 2, 4, 8 or 16 bits), RGB (8 or 16), palette
(1, 2, 4 or 8), gray + alpha and RGBA (8 or 16), Adam7-interlaced or not -- what OpenSlide's RGBA `read_region` tiles,
viewer exports, quantised or binarised masks and scanners' 16-bit exports are saved as.  Gray is copied to R, G and B
(1 / 2 / 4-bit samples scaled by 255 / 85 / 17), alpha is dropped (not composited), tRNS is ignored, a 16-bit sample
becomes its high byte, and a palette index past the last PLTE entry gives black.  The one difference from Pillow is
16-bit grayscale, which Pillow opens as "I;16" and clips to 255 where this decoder takes the high byte; whether
TensorFlow takes the high byte or rescales 16-bit samples is not verified.  8-bit RGB tiles decode to the same bytes
with the option as without it.  A palette image without PLTE, a PLTE of 0 or more than 256 entries or a length that
is not a multiple of 3, and an illegal colour type / bit depth pair raise ValueError naming the tile before the GPU
runs.
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
    offsets: n + 1 non-decreasing int64 byte offsets (host).
    convert_rgb: accept every colour type, bit depth and interlace and convert to RGB8 (module docstring); the
    default accepts 8-bit RGB non-interlaced tiles only."""

    FORMAT = "png"
    PARSE_OPTIONS = True

    def __init__(self, data, offsets, convert_rgb: bool = False):
        if not isinstance(convert_rgb, (bool, np.bool_)):
            raise ValueError(f"convert_rgb must be a bool, got {convert_rgb!r}")
        super().__init__(data, offsets)
        self.convert_rgb = bool(convert_rgb)

    @property
    def flags(self) -> int | None:
        # without the option: None, so the batch goes through the entry points without flags, as before the option
        return _ffi.BQ_PNG_CONVERT_RGB if self.convert_rgb else None

    def options(self) -> dict:
        return dict(convert_rgb=self.convert_rgb)


def status_message(code: int) -> str:
    return encoded.status_message("png", code)


def inspect(batch: PngBatch, px: int = nature2022.tile_px) -> np.ndarray:
    """Host chunk parse of every tile under the batch's decode option, no GPU needed: int32 status per tile (0 =
    accepted, else a BQ_PNG_* code, see `status_message`)."""
    return encoded.inspect("png", batch, px)


def check(batch: PngBatch, px: int = nature2022.tile_px) -> None:
    """raise ValueError for the first tile `decode` would reject by its headers"""
    return encoded.check("png", batch, px)


def decode(batch: PngBatch, px: int = nature2022.tile_px, ctx: _ffi.Context | None = None, out=None):
    """uint8 NHWC [n, px, px, 3] tiles decoded on the GPU with the batch's decode option.  `out` may be a preallocated numpy array or CUDA torch tensor
    of that shape (device output stays on the device); default: a new numpy array."""
    return encoded.decode("png", batch, px, ctx, out)
