"""Compressed test inputs (test only): JPEG tiles written by Pillow (libjpeg-turbo), the Pillow decode that is the GPU
decoder's contract, tiles that drive the decoder's clamps, and a TFRecord writer for Slideflow-style tile records."""
from __future__ import annotations

import numpy as np

from .synth import TILE_PX

SUBSAMPLING = {"4:4:4": 0, "4:2:2": 1, "4:2:0": 2}


def degenerate_tiles(px=TILE_PX):
    """tiles that drive the decoder's clamps: constant grey, all 0, all 255, a 1-pixel checkerboard, saturated chroma"""
    grey = np.full((px, px, 3), 128, np.uint8)
    zero = np.zeros((px, px, 3), np.uint8)
    full = np.full((px, px, 3), 255, np.uint8)
    cb = ((np.indices((px, px)).sum(0) % 2) * 255).astype(np.uint8)
    checker = np.stack([cb] * 3, -1)
    sat = np.zeros((px, px, 3), np.uint8)
    sat[..., 0] = 255
    sat[::2, :, 2] = 255
    sat[:, ::3, 1] = 255
    return np.stack([grey, zero, full, checker, sat])


def jpeg_encode(tile, quality=90, subsampling="4:2:0", optimize=False, restart_blocks=None, restart_rows=None,
                progressive=False, mode="RGB"):
    """one tile as JPEG bytes written by Pillow (libjpeg-turbo)"""
    import io

    from PIL import Image, ImageFile
    kw = dict(quality=quality, subsampling=SUBSAMPLING[subsampling], optimize=optimize, progressive=progressive)
    if restart_blocks:
        kw["restart_marker_blocks"] = restart_blocks
    if restart_rows:
        kw["restart_marker_rows"] = restart_rows
    img = Image.fromarray(tile)
    if mode != "RGB":
        img = img.convert(mode)
    old = ImageFile.MAXBLOCK
    ImageFile.MAXBLOCK = max(old, 4 * tile.size)   # optimize=True encodes in one buffer; quality 100 4:4:4 exceeds Pillow's guess
    try:
        bio = io.BytesIO()
        img.save(bio, "JPEG", **kw)
    finally:
        ImageFile.MAXBLOCK = old
    return bio.getvalue()


def pil_decode(b):
    """the decode contract: what Pillow's libjpeg-turbo returns"""
    import io

    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))


def _crc32c(b: bytes) -> int:
    table = _crc32c.table if hasattr(_crc32c, "table") else None
    if table is None:
        table = []
        for i in range(256):
            c = i
            for _ in range(8):
                c = (c >> 1) ^ (0x82F63B78 if c & 1 else 0)
            table.append(c)
        _crc32c.table = table
    c = 0xFFFFFFFF
    for x in b:
        c = (c >> 8) ^ table[(c ^ x) & 0xFF]
    return c ^ 0xFFFFFFFF


def masked_crc32c(b: bytes) -> int:
    c = _crc32c(b)
    return ((((c >> 15) | (c << 17)) & 0xFFFFFFFF) + 0xA282EAD8) & 0xFFFFFFFF


def _varint(v: int) -> bytes:
    out = bytearray()
    v &= (1 << 64) - 1
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _ld(field: int, payload: bytes) -> bytes:
    return _varint(field << 3 | 2) + _varint(len(payload)) + payload


def tf_example(features: dict, order=None, packed=True, extra_unknown=False) -> bytes:
    """tf.train.Example bytes: values are bytes (bytes_list), int (int64_list) or float (float_list)"""
    entries = []
    for k in (order or list(features)):
        v = features[k]
        if isinstance(v, (bytes, bytearray)):
            feat = _ld(1, _ld(1, bytes(v)))
        elif isinstance(v, float):
            feat = _ld(2, _ld(1, np.float32(v).tobytes()))
        elif packed:
            feat = _ld(3, _ld(1, _varint(int(v))))
        else:
            feat = _ld(3, _varint(1 << 3 | 0) + _varint(int(v)))
        entry = _ld(1, k.encode()) + _ld(2, feat)
        if extra_unknown:
            entry = _varint(7 << 3 | 0) + _varint(5) + entry      # unknown varint field inside the map entry
        entries.append(_ld(1, entry))
    body = _ld(1, b"".join(entries))
    if extra_unknown:
        body = _ld(9, b"unknown") + body + _varint(10 << 3 | 5) + b"\0\0\0\0"
    return body


def tfrecord_frame(payload: bytes) -> bytes:
    n = len(payload).to_bytes(8, "little")
    return (n + masked_crc32c(n).to_bytes(4, "little") + payload + masked_crc32c(payload).to_bytes(4, "little"))


def write_tfrecord(path, images, slides, locs=None):
    """Slideflow-style tile records: image_raw (JPEG bytes), slide (UTF-8), loc_x, loc_y"""
    with open(path, "wb") as f:
        for i, (img, slide) in enumerate(zip(images, slides)):
            feats = {"image_raw": img, "slide": slide.encode("utf-8")}
            if locs is not None:
                feats["loc_x"], feats["loc_y"] = int(locs[i][0]), int(locs[i][1])
            f.write(tfrecord_frame(tf_example(feats)))
