"""numpy restatement of the decode options TensorFlow's decode_jpeg exposes (test oracle only), on top of
oracle/jpeg_ref.py's marker parse, Huffman stage, fancy upsampling and YCbCr -> RGB:

  * dct_method "INTEGER_FAST" (and "", which TensorFlow maps to it): libjpeg-turbo's JDCT_IFAST IDCT (jidctfst.c, 8-bit
    samples, no accurate rounding) with jddctmgr.c's multiplier table;
  * fancy_upscaling=False: 4:2:2 / 4:2:0 chroma replicated (jdmerge.c's merged upsampler), not interpolated.

`pil_decode_fast(b)` is the libjpeg-turbo decode these are pinned to: Pillow's draft decode, which asks libjpeg-turbo
for JDCT_FASTEST (= JDCT_IFAST) and turns fancy upsampling off.
"""
from __future__ import annotations

import numpy as np

from oracle import jpeg_ref, jpeg_synth
from oracle.synth import TILE_PX

DCT_METHODS = {"INTEGER_ACCURATE": "INTEGER_ACCURATE", "INTEGER_FAST": "INTEGER_FAST", "": "INTEGER_FAST"}

# jddctmgr.c aanscales: 16384 * s(row) * s(col), s(0) = 1, s(k) = sqrt(2) cos(k pi / 16), rounded
AAN = np.array([
    16384, 22725, 21407, 19266, 16384, 12873, 8867, 4520,
    22725, 31521, 29692, 26722, 22725, 17855, 12299, 6270,
    21407, 29692, 27969, 25172, 21407, 16819, 11585, 5906,
    19266, 26722, 25172, 22654, 19266, 15137, 10426, 5315,
    16384, 22725, 21407, 19266, 16384, 12873, 8867, 4520,
    12873, 17855, 16819, 15137, 12873, 10114, 6967, 3552,
    8867, 12299, 11585, 10426, 8867, 6967, 4799, 2446,
    4520, 6270, 5906, 5315, 4520, 3552, 2446, 1247], np.int64)


def ifast_multipliers(q: np.ndarray) -> np.ndarray:
    """jddctmgr.c: the IFAST dequantisation multiplier of each table entry (natural order), IFAST_MULT_TYPE = int16"""
    return ((q.astype(np.int64) * AAN + 2048) >> 12).astype(np.int16).astype(np.int64)


def idct_ifast(coef: np.ndarray, q: np.ndarray) -> np.ndarray:
    """jidctfst.c jpeg_idct_ifast on blocks [..., 64] (natural order) -> uint8 [..., 8, 8].  Multiplies truncate
    (CONST_BITS 8); the column pass keeps its scale, the row pass output is shifted right by 5 (PASS1_BITS + 3); the
    range limit saturates to [0, 255] after +128, as libjpeg-turbo's SIMD IDCT does."""
    x = (coef.astype(np.int64) * ifast_multipliers(q)).reshape(coef.shape[:-1] + (8, 8))

    def mul(v, c):
        return (v * c) >> 8

    def one_pass(v):                  # v[..., 8 (along the transform), m]
        i0, i1, i2, i3, i4, i5, i6, i7 = (v[..., k, :] for k in range(8))
        t10, t11, t13 = i0 + i4, i0 - i4, i2 + i6
        t12 = mul(i2 - i6, 362) - t13
        e0, e3, e1, e2 = t10 + t13, t10 - t13, t11 + t12, t11 - t12
        z13, z10, z11, z12 = i5 + i3, i5 - i3, i1 + i7, i1 - i7
        o7 = z11 + z13
        o11 = mul(z11 - z13, 362)
        z5 = mul(z10 + z12, 473)
        o10 = mul(z12, 277) - z5
        o12 = mul(z10, -669) + z5
        o6 = o12 - o7
        o5 = o11 - o6
        o4 = o10 + o5
        return np.stack([e0 + o7, e1 + o6, e2 + o5, e3 - o4, e3 + o4, e2 - o5, e1 - o6, e0 - o7], axis=-2)

    ws = one_pass(x)
    ws = np.swapaxes(one_pass(np.swapaxes(ws, -1, -2)), -1, -2) >> 5
    return np.clip(ws + 128, 0, 255).astype(np.uint8)


def _replicate(p, fh, fv):
    return np.repeat(np.repeat(p, fv, 0), fh, 1)


def decode(b: bytes, dct_method: str = "INTEGER_ACCURATE", fancy_upscaling: bool = True) -> np.ndarray:
    """jpeg_ref.decode with TensorFlow's decode_jpeg options; the defaults are jpeg_ref.decode itself"""
    if dct_method not in DCT_METHODS:
        raise ValueError(f"dct_method must be one of {sorted(DCT_METHODS)}, got {dct_method!r}")
    idct = idct_ifast if DCT_METHODS[dct_method] == "INTEGER_FAST" else jpeg_ref.idct_islow
    hdr = jpeg_ref.parse(b)
    coef, (mcux, mcuy, hmax, vmax) = jpeg_ref.coefficients(hdr, b)
    pl = []
    for c, blocks in zip(hdr["comps"], coef):
        px = idct(blocks, hdr["qt"][c["tq"]])                       # [by, bx, 8, 8]
        by, bx = px.shape[:2]
        pl.append(px.transpose(0, 2, 1, 3).reshape(by * 8, bx * 8))
    H, W = hdr["height"], hdr["width"]
    full = [pl[0][:H, :W]]
    for c, p in zip(hdr["comps"][1:], pl[1:]):
        dh, dw = -(-H * c["v"] // vmax), -(-W * c["h"] // hmax)
        p = p[:dh, :dw]
        fh, fv = hmax // c["h"], vmax // c["v"]
        if (fh, fv) != (1, 1):
            if not fancy_upscaling:
                p = _replicate(p, fh, fv)
            elif (fh, fv) == (2, 2):
                p = jpeg_ref._fancy_h2v2(p)
            else:
                p = jpeg_ref._fancy_h2v1(p)
        full.append(p[:H, :W])
    return jpeg_ref.ycc_to_rgb(*full)


def pil_decode_fast(b: bytes) -> np.ndarray:
    """libjpeg-turbo's JDCT_IFAST decode with chroma replicated, through Pillow.  Pillow's JPEG decoder arguments are
    (rawmode, jpegmode, scale, draft); with draft set it asks libjpeg-turbo for dct_method = JDCT_FASTEST (JDCT_IFAST)
    and do_fancy_upsampling = FALSE, so 4:2:x tiles go through the merged upsampler.  Scale 1 keeps the full size."""
    import io

    from PIL import Image
    im = Image.open(io.BytesIO(b))
    d, e, o, _ = im.tile[0]
    im.tile = [(d, e, o, ("RGB", "", 1, 1))]
    return np.asarray(im.convert("RGB"))


# ------------------------------------------------------------------------------------------------------------------
# test inputs
# ------------------------------------------------------------------------------------------------------------------
def saturated_tiles(px=TILE_PX):
    """pure primaries at pixel pitch: an R/B checkerboard, G / black stripes and R, G, B columns"""
    yy, xx = np.indices((px, px))
    prim = (np.eye(3) * 255).astype(np.uint8)
    return np.stack([prim[np.where((yy + xx) % 2, 0, 2)], prim[1] * (xx % 2 == 0)[..., None].astype(np.uint8),
                     prim[xx % 3]])


def dqt16_encode(tile, subsampling, restart=None):
    """a tile with 16-bit quantisation tables (Pq = 1): entries 200 ... 20063, the largest at low frequencies in the
    chroma table, where the IFAST multiplier overflows its int16 type"""
    import io

    from PIL import Image
    lum = np.linspace(200, 20063, 64).astype(int).tolist()
    kw = dict(qtables=[lum, lum[::-1]], subsampling=jpeg_synth.SUBSAMPLING[subsampling])
    if restart:
        kw["restart_marker_blocks"] = restart
    bio = io.BytesIO()
    Image.fromarray(tile).save(bio, "JPEG", **kw)
    return bio.getvalue()
