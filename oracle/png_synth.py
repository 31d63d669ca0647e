"""PNG test inputs (test only): a PNG writer built from zlib + struct with control over every part the GPU decoder
reads (filter per row, zlib level / strategy / window / flushes, IDAT chunk sizes, ancillary chunks), Pillow's own PNG
encoding, the Pillow decode that is the decoder's contract, and a small DEFLATE bit-writer for streams zlib must
reject."""
from __future__ import annotations

import struct
import zlib

import numpy as np

from .synth import TILE_PX

SIGNATURE = b"\x89PNG\r\n\x1a\n"
STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "rle": zlib.Z_RLE,
              "huffman": zlib.Z_HUFFMAN_ONLY, "fixed": zlib.Z_FIXED}


def chunk(kind: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + kind + data + struct.pack(">I", zlib.crc32(kind + data))


def ihdr(w, h, depth=8, colour=2, interlace=0, compression=0, filt=0) -> bytes:
    return chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, colour, compression, filt, interlace))


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(tile, filters) -> bytes:
    """the filtered scanlines of an RGB tile: filters = one type 0-4 per row"""
    h, w, _ = tile.shape
    raw = tile.reshape(h, w * 3).astype(np.int32)
    out = bytearray()
    for r in range(h):
        x = raw[r]
        up = raw[r - 1] if r else np.zeros_like(x)
        left = np.concatenate([np.zeros(3, np.int32), x[:-3]])
        ul = np.concatenate([np.zeros(3, np.int32), up[:-3]])
        ft = int(filters[r])
        pred = [np.zeros_like(x), left, up, (left + up) >> 1, _paeth(left, up, ul)][ft]
        out.append(ft)
        out += ((x - pred) & 255).astype(np.uint8).tobytes()
    return bytes(out)


def zlib_stream(raw: bytes, level=6, strategy="default", wbits=15, flush=None, row_bytes=None) -> bytes:
    """zlib stream of `raw`; flush = "sync" (Z_SYNC_FLUSH after every row) or "full" (Z_FULL_FLUSH every 7 rows)"""
    co = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, STRATEGIES[strategy])
    if flush is None:
        return co.compress(raw) + co.flush()
    mode, every = (zlib.Z_SYNC_FLUSH, 1) if flush == "sync" else (zlib.Z_FULL_FLUSH, 7)
    out = []
    rows = [raw[i:i + row_bytes] for i in range(0, len(raw), row_bytes)]
    for i, r in enumerate(rows):
        out.append(co.compress(r))
        if (i + 1) % every == 0:
            out.append(co.flush(mode))
    out.append(co.flush())
    return b"".join(out)


def assemble(w, h, zdata: bytes, idat_size=None, before=(), after=(), header=None) -> bytes:
    """signature, IHDR, chunks `before`, IDAT (split into payloads of idat_size bytes), chunks `after`, IEND"""
    step = idat_size or max(1, len(zdata))
    idats = [chunk(b"IDAT", zdata[i:i + step]) for i in range(0, max(1, len(zdata)), step)]
    return (SIGNATURE + (header if header is not None else ihdr(w, h)) + b"".join(before) + b"".join(idats)
            + b"".join(after) + chunk(b"IEND", b""))


def ancillary(iccp_bytes=0, seed=0) -> list:
    """tEXt, pHYs, sRGB / gAMA and (when iccp_bytes) an iCCP chunk of about that size"""
    out = [chunk(b"tEXt", b"Comment\0synthetic tile"), chunk(b"pHYs", struct.pack(">IIB", 3937, 3937, 1)),
           chunk(b"gAMA", struct.pack(">I", 45455))]
    if iccp_bytes:
        rng = np.random.default_rng(seed)
        prof = zlib.compress(rng.integers(0, 256, iccp_bytes, dtype=np.uint8).tobytes(), 0)
        out.append(chunk(b"iCCP", b"icc\0\0" + prof))
    return out


def png_encode(tile, filters=0, level=6, strategy="default", wbits=15, flush=None, idat_size=None, before=(), after=(),
               seed=0) -> bytes:
    """tile as PNG: filters = one type 0-4 for every row, "random" (a random type per row) or a per-row sequence"""
    h, w, _ = tile.shape
    if isinstance(filters, str):
        filters = np.random.default_rng(seed).integers(0, 5, h)
    elif np.isscalar(filters):
        filters = [filters] * h
    raw = filter_rows(tile, filters)
    z = zlib_stream(raw, level, strategy, wbits, flush, 1 + 3 * w)
    return assemble(w, h, z, idat_size, before, after)


def pil_encode(tile, compress_level=6, mode="RGB") -> bytes:
    import io

    from PIL import Image
    img = Image.fromarray(tile)
    if mode != "RGB":
        img = img.convert(mode)
    bio = io.BytesIO()
    img.save(bio, "PNG", compress_level=compress_level)
    return bio.getvalue()


def pil_decode(b):
    """the decode contract: what Pillow returns"""
    import io

    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))


def encodings():
    """(label, png_encode keyword arguments) of the writer matrix: every filter type, zlib levels 0-9, every strategy,
    a 512-byte window, sync / full flushes, IDAT payloads of 1, 7, 8192 and 65536 bytes, ancillary chunks before and
    after IDAT including a 3 KB iCCP"""
    out = [(f"filter {f}", dict(filters=f)) for f in (0, 1, 2, 3, 4, "random")]
    out += [(f"level {k}", dict(filters="random", level=k)) for k in range(10)]
    out += [(f"strategy {k}", dict(filters="random", strategy=k)) for k in STRATEGIES if k != "default"]
    out += [("wbits 9", dict(filters="random", wbits=9, level=9)), ("wbits 9 rle", dict(filters=2, wbits=9, strategy="rle"))]
    out += [("sync flush every row", dict(filters="random", flush="sync")),
            ("full flush every 7 rows", dict(filters=4, flush="full", level=1))]
    out += [(f"IDAT {n} bytes", dict(filters="random", idat_size=n)) for n in (1, 7, 8192, 65536)]
    out += [("ancillary chunks + iCCP", dict(filters="random", before=ancillary(3000), after=ancillary()))]
    return out


PIL_LEVELS = (1, 6, 9)


def distance_tile(px=TILE_PX, period=36, seed=0):
    """random rows where row r repeats row r - period: with filter 0 the matches lie period * (1 + 3 px) bytes back
    (32,328 at 299 px), near the 32 KB window limit"""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 256, (px, px, 3), dtype=np.uint8)
    for r in range(period, px):
        t[r] = t[r - period]
    return t


def zlib_wrap(deflate: bytes, raw: bytes, cinfo=7) -> bytes:
    """zlib header (window 2**(cinfo + 8)) + DEFLATE data + Adler-32 of raw"""
    cmf = cinfo << 4 | 8
    flg = 31 - (cmf << 8) % 31
    return bytes([cmf, flg]) + deflate + struct.pack(">I", zlib.adler32(raw))


# ------------------------------------------------------------------------------------------------------------------
# DEFLATE bit-writer for hand-made (mostly invalid) streams
# ------------------------------------------------------------------------------------------------------------------
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227,
            258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
             4097, 6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [i // 2 for i in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


def canonical(lengths):
    """{symbol: (code, length)} of a canonical Huffman code (RFC 1951 3.2.2)"""
    count = [0] * 16
    for n in lengths:
        count[n] += 1
    count[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    out = {}
    for s, n in enumerate(lengths):
        if n:
            out[s] = (nxt[n], n)
            nxt[n] += 1
    return out


FIXED_LIT = canonical([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8)
FIXED_DIST = canonical([5] * 32)


class BitWriter:
    def __init__(self):
        self.bits = []

    def put(self, value, n):           # an n-bit field, LSB first
        self.bits += [(value >> i) & 1 for i in range(n)]

    def code(self, code, n):           # a Huffman code, MSB first
        self.bits += [(code >> (n - 1 - i)) & 1 for i in range(n)]

    def align(self):
        self.bits += [0] * (-len(self.bits) % 8)

    def bytes(self):
        self.align()
        return np.packbits(np.asarray(self.bits, np.uint8), bitorder="little").tobytes()


def put_length(bw, lit, length):
    s = max(i for i, b in enumerate(LEN_BASE) if b <= length)
    if length == 258:
        s = 28
    bw.code(*lit[257 + s])
    bw.put(length - LEN_BASE[s], LEN_EXTRA[s])


def put_dist(bw, dist_code, dist):
    s = max(i for i, b in enumerate(DIST_BASE) if b <= dist)
    bw.code(*dist_code[s])
    bw.put(dist - DIST_BASE[s], DIST_EXTRA[s])


def fixed_block(bw, tokens, final=True):
    """tokens: ints (literal bytes), ("match", length, distance), ("sym", literal/length symbol) or ("dsym", distance
    symbol)"""
    bw.put(int(final), 1)
    bw.put(1, 2)
    for t in tokens:
        if isinstance(t, tuple) and t[0] == "match":
            put_length(bw, FIXED_LIT, t[1])
            put_dist(bw, FIXED_DIST, t[2])
        elif isinstance(t, tuple):
            bw.code(*(FIXED_LIT if t[0] == "sym" else FIXED_DIST)[t[1]])
        else:
            bw.code(*FIXED_LIT[int(t)])
    bw.code(*FIXED_LIT[256])


def dynamic_header(bw, lit_lens, dist_lens, final=True, cl_symbols=None):
    """dynamic block header: the code-length code gives 0..15 length 4 (complete); cl_symbols overrides the
    code-length symbol sequence with (symbol, extra value) pairs, then symbols 16 / 17 / 18 get codes too"""
    bw.put(int(final), 1)
    bw.put(2, 2)
    if cl_symbols is None:
        cl_lens = [4] * 16 + [0, 0, 0]
        cl_symbols = [(n, 0) for n in list(lit_lens) + list(dist_lens)]
    else:
        cl_lens = [4] * 14 + [0, 0, 5, 5, 4]        # 0..13 and 18 length 4, 16 / 17 length 5
    bw.put(len(lit_lens) - 257, 5)
    bw.put(len(dist_lens) - 1, 5)
    bw.put(19 - 4, 4)
    for s in CL_ORDER:
        bw.put(cl_lens[s], 3)
    cl = canonical(cl_lens)
    for s, extra in cl_symbols:
        bw.code(*cl[s])
        if s >= 16:
            bw.put(extra, {16: 2, 17: 3, 18: 7}[s])


def literal_dynamic_code():
    """a complete literal/length code (0..253 length 8; 254, 255, 256, 257 length 9) and a single distance code"""
    return [8] * 254 + [9] * 4, [1]


def _literal_dynamic_block(bw, data, final=True):
    lit_lens, dist_lens = literal_dynamic_code()
    dynamic_header(bw, lit_lens, dist_lens, final)
    code = canonical(lit_lens)
    for b in data:
        bw.code(*code[b])
    bw.code(*code[256])


def crafted_streams(raw: bytes, row_bytes: int):
    """Hand-made zlib streams around the filtered image `raw`: name -> (stream, the GPU decoder's status message, whether
    zlib.decompress accepts it, the bytes it then returns).  A GPU status of None means the tile decodes."""
    out = {}

    def fixed(tokens, cinfo=7, data=raw):
        bw = BitWriter()
        fixed_block(bw, tokens)
        return zlib_wrap(bw.bytes(), data, cinfo)

    def dynamic(lit_lens, dist_lens, cl_symbols=None):
        bw = BitWriter()
        dynamic_header(bw, lit_lens, dist_lens, True, cl_symbols)
        return zlib_wrap(bw.bytes(), raw)

    bw = BitWriter()
    bw.put(1, 1)
    bw.put(3, 2)
    out["block type 3"] = (zlib_wrap(bw.bytes(), raw), "bad block")
    bw = BitWriter()
    bw.put(1, 1)
    bw.put(0, 2)
    bw.align()
    bw.put(5, 16)
    bw.put(5, 16)
    out["stored LEN != ~NLEN"] = (zlib_wrap(bw.bytes() + b"abcde", raw), "bad block")
    out["literal/length symbol 286"] = (fixed([0, ("sym", 286)]), "bad Huffman code")
    out["literal/length symbol 287"] = (fixed([0, ("sym", 287)]), "bad Huffman code")
    out["distance code 30"] = (fixed([0, ("sym", 257), ("dsym", 30)]), "bad Huffman code")
    out["distance before the stream"] = (fixed([0, ("match", 3, 2)]), "bad distance")
    out["over-subscribed code"] = (dynamic([8] * 257, [1]), "bad Huffman code")
    out["incomplete code"] = (dynamic([8] * 128 + [0] * 128 + [8], [1]), "bad Huffman code")
    out["repeat with no previous length"] = (dynamic([8] * 257, [1], [(16, 0)] + [(8, 0)] * 257), "bad Huffman code")
    out["no end-of-block code"] = (dynamic([8] * 256 + [0], [1]), "bad Huffman code")
    out["too many length symbols"] = (dynamic([8] * 254 + [9] * 4 + [0] * 29, [1]), "bad Huffman code")
    # valid: an empty dynamic block whose literal/length code is one code of length 1 (zlib's single-code case) and
    # which has no distance code, then every byte as a literal of a complete dynamic code
    bw = BitWriter()
    dynamic_header(bw, [0] * 256 + [1], [0], final=False)
    bw.code(*canonical([0] * 256 + [1])[256])
    _literal_dynamic_block(bw, raw)
    out["single-code block, then dynamic literals"] = (zlib_wrap(bw.bytes(), raw), None)
    # valid: a match 1000 bytes back under a zlib header declaring a 512-byte window
    far = raw[:2 * row_bytes + 200] + raw[row_bytes + 100:row_bytes + 110] + raw[2 * row_bytes + 210:]
    out["distance beyond the declared window"] = (
        fixed(list(far[:2 * row_bytes + 200]) + [("match", 10, row_bytes + 100)] + list(far[2 * row_bytes + 210:]),
              cinfo=1, data=far), None)
    good = zlib.compress(raw, 6)
    out["truncated stream"] = (good[:len(good) // 2], "truncated data")
    out["no Adler-32"] = (good[:-4], "truncated data")
    out["Adler-32 flipped"] = (good[:-1] + bytes([good[-1] ^ 1]), "Adler-32 mismatch")
    out["one byte short"] = (zlib.compress(raw[:-1]), "wrong decompressed size")
    out["three bytes long"] = (zlib.compress(raw + b"\0\0\0"), "wrong decompressed size")
    bad = bytearray(raw)
    bad[5 * row_bytes] = 5
    out["filter type 5"] = (zlib.compress(bytes(bad)), "bad filter type")
    res = {}
    for k, (z, status) in out.items():
        try:
            got = zlib.decompress(z)
        except zlib.error:
            got = None
        res[k] = (z, status, got)
    return res
