"""Slideflow tile TFRecords read without TensorFlow (csrc/tfrecord.cu).

Each record is a `tf.train.Example` holding one JPEG or PNG tile and where it came from.  `read(paths)` verifies both
CRCs of every record and returns the tiles as one `jpeg.JpegBatch` or `png.PngBatch` (decoded on the GPU by `predict` /
`jpeg.decode` / `png.decode`) with the slide name and tile location of each.  The feature keys default to Slideflow's
(`image_raw`, `slide`, `loc_x`, `loc_y`).  Compressed (gzip / zlib) record files are rejected: decompress them first.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _ffi
from .jpeg import JpegBatch
from .png import SIGNATURE as PNG_SIGNATURE
from .png import PngBatch

LOC_MISSING = np.iinfo(np.int64).min


def scan(buf, image_key="image_raw", slide_key="slide", x_key="loc_x", y_key="loc_y"):
    """Records of one TFRecord file held in memory: (image [n, 2], slide [n, 2], loc [n, 2]) int64 arrays, the byte
    ranges [begin, end) of the image and slide values in `buf` (slide -1 when absent) and (loc_x, loc_y)
    (`LOC_MISSING` when absent).  Raises ValueError on a bad CRC, a truncated record or a malformed Example."""
    buf = np.frombuffer(buf, np.uint8) if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf, np.uint8)
    lib = _ffi.load_library()
    keys = [k.encode() if k is not None else None for k in (image_key, slide_key, x_key, y_key)]
    cap = max(16, buf.size // 4096)
    err = C.create_string_buffer(512)
    while True:
        image, slide, loc = (np.empty((cap, 2), np.int64) for _ in range(3))
        n = C.c_int64(0)
        rc = lib.bq_tfrecord_scan(_ffi.ptr(buf), buf.size, *keys, cap, C.byref(n), _ffi.ptr(image), _ffi.ptr(slide),
                                  _ffi.ptr(loc), err, len(err))
        if rc == _ffi.BQ_ERR_DATA:
            raise ValueError(err.value.decode(errors="replace"))
        if rc != 0:
            raise ValueError("bq_tfrecord_scan: bad argument")
        if n.value <= cap:
            k = n.value
            return image[:k], slide[:k], loc[:k]
        cap = n.value


def read(paths, image_key="image_raw", slide_key="slide", x_key="loc_x", y_key="loc_y"):
    """(batch, slides, loc_x, loc_y) over the records of `paths` (one path or a list), in file order.
    batch: a PngBatch when every image starts with the PNG signature, else a JpegBatch (whatever is not JPEG then fails
    in the JPEG decoder, naming the tile).  A set that mixes PNG with other images raises ValueError naming the first
    record (file, index in the file) whose format differs from record 0.  slides: list of str (UTF-8); loc_x / loc_y:
    int64 arrays."""
    if isinstance(paths, (str, os.PathLike)):
        paths = [paths]
    parts, sizes, slides, locs = [], [], [], []
    first_png = None
    for p in paths:
        with open(p, "rb") as f:
            buf = np.frombuffer(f.read(), np.uint8)
        image, slide, loc = scan(buf, image_key, slide_key, x_key, y_key)
        for r, ((a, b), (sa, sb)) in enumerate(zip(image, slide)):
            is_png = buf[a:min(b, a + len(PNG_SIGNATURE))].tobytes() == PNG_SIGNATURE
            if first_png is None:
                first_png = is_png
            elif is_png != first_png:
                kinds = ("PNG", "not PNG") if first_png else ("not PNG", "PNG")
                raise ValueError(f"{os.fspath(p)} record {r}: image is {kinds[1]} but the first record's is {kinds[0]}; "
                                 "a record set must hold one image format")
            parts.append(buf[a:b])
            sizes.append(b - a)
            slides.append(buf[sa:sb].tobytes().decode("utf-8") if sa >= 0 else "")
        locs.append(loc)
    offsets = np.zeros(len(sizes) + 1, np.int64)
    offsets[1:] = np.cumsum(sizes)
    data = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    loc = np.concatenate(locs) if locs else np.zeros((0, 2), np.int64)
    return (PngBatch if first_png else JpegBatch)(data, offsets), slides, loc[:, 0].copy(), loc[:, 1].copy()


def crc32c(b) -> int:
    return int(_ffi.load_library().bq_crc32c(_ffi.ptr(np.frombuffer(bytes(b), np.uint8)), len(b)))


def masked_crc32c(b) -> int:
    return int(_ffi.load_library().bq_crc32c_masked(_ffi.ptr(np.frombuffer(bytes(b), np.uint8)), len(b)))
