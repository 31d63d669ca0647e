"""Test-only reference for the PNG decode option `convert_rgb`: a writer for every colour type, bit depth and interlace
of the PNG specification (filter type per row 0-4 or random), and a numpy decoder that restates the decode contract --
`zlib.decompress` for the stream, then the unfilter, the Adam7 deinterlace and the conversion to RGB8:

- gray is copied to R, G and B; 1 / 2 / 4-bit samples are scaled by 255 / 85 / 17 (libpng's expand_gray_1_2_4_to_8);
- alpha (colour types 4 and 6) is dropped, tRNS ignored;
- a 16-bit sample becomes its high byte (libpng's strip_16);
- a palette index at or past the number of PLTE entries gives black."""
from __future__ import annotations

import struct
import zlib

import numpy as np

from oracle.png_synth import SIGNATURE, chunk, ihdr

# the legal (colour type, bit depth) pairs
DEPTHS = {0: (1, 2, 4, 8, 16), 2: (8, 16), 3: (1, 2, 4, 8), 4: (8, 16), 6: (8, 16)}
COMBOS = [(c, d) for c, ds in DEPTHS.items() for d in ds]
CHANNELS = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}
NAMES = {0: "gray", 2: "RGB", 3: "palette", 4: "gray+alpha", 6: "RGBA"}
ADAM7 = [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)]
FILTER_MODES = (0, 1, 2, 3, 4, "random")


def label(colour, depth, interlace=0) -> str:
    return f"{NAMES[colour]} {depth}-bit{' Adam7' if interlace else ''}"


def passes(w, h, interlace):
    """(pass index, x0, y0, dx, dy, pass width, pass height) of every non-empty pass, in stream order"""
    for p, (x0, y0, dx, dy) in enumerate(ADAM7 if interlace else [(0, 0, 1, 1)]):
        pw, ph = max(0, (w - x0 + dx - 1) // dx), max(0, (h - y0 + dy - 1) // dy)
        if pw and ph:
            yield p, x0, y0, dx, dy, pw, ph


def bpp(colour, depth) -> int:
    return max(1, CHANNELS[colour] * depth // 8)


def row_bytes(w, colour, depth) -> int:
    """filtered row length of a row `w` pixels wide, filter byte included"""
    return 1 + (w * CHANNELS[colour] * depth + 7) // 8


def pack(samples, depth) -> np.ndarray:
    """samples [h, w, ch] -> packed rows [h, nbytes] (16-bit big-endian, sub-byte MSB first, zero-padded)"""
    h, w, ch = samples.shape
    s = samples.reshape(h, w * ch).astype(np.uint16)
    if depth == 16:
        return s.astype(">u2").view(np.uint8).reshape(h, 2 * w * ch)
    if depth == 8:
        return s.astype(np.uint8)
    bits = ((s[..., None] >> np.arange(depth - 1, -1, -1)) & 1).astype(np.uint8).reshape(h, -1)
    return np.packbits(bits, axis=1)


def unpack(rows, w, ch, depth) -> np.ndarray:
    """packed rows [h, nbytes] -> samples [h, w, ch] (uint16)"""
    h = rows.shape[0]
    if depth == 16:
        return rows[:, :2 * w * ch].copy().view(">u2").astype(np.uint16).reshape(h, w, ch)
    if depth == 8:
        return rows[:, :w * ch].astype(np.uint16).reshape(h, w, ch)
    bits = np.unpackbits(rows, axis=1)[:, :w * ch * depth].reshape(h, w * ch, depth).astype(np.uint16)
    return (bits << np.arange(depth - 1, -1, -1, dtype=np.uint16)).sum(-1).astype(np.uint16).reshape(h, w, ch)


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(rows, filters, unit) -> bytes:
    """packed rows [h, n] -> filtered stream: filters = one type 0-4 per row"""
    out = bytearray()
    prev = np.zeros(rows.shape[1], np.int32)
    for r in range(rows.shape[0]):
        x = rows[r].astype(np.int32)
        left = np.concatenate([np.zeros(unit, np.int32), x[:-unit]])[:len(x)]
        ul = np.concatenate([np.zeros(unit, np.int32), prev[:-unit]])[:len(x)]
        ft = int(filters[r])
        pred = [np.zeros_like(x), left, prev, (left + prev) >> 1, _paeth(left, prev, ul)][ft]
        out.append(ft)
        out += ((x - pred) & 255).astype(np.uint8).tobytes()
        prev = x
    return bytes(out)


def unfilter(data: bytes, h, n, unit) -> np.ndarray:
    """filtered stream of h rows of n bytes (after their filter byte) -> packed rows [h, n]; ValueError on a filter
    type > 4"""
    out = np.zeros((h, n), np.uint8)
    prev = bytearray(n)
    for r in range(h):
        ft = data[r * (n + 1)]
        f = data[r * (n + 1) + 1:(r + 1) * (n + 1)]
        if ft > 4:
            raise ValueError(f"bad filter type {ft} in row {r}")
        if ft == 0:
            cur = bytearray(f)
        elif ft == 1:
            a = np.frombuffer(f, np.uint8).astype(np.int64)
            pad = (-n) % unit
            a = np.concatenate([a, np.zeros(pad, np.int64)]).reshape(-1, unit)
            cur = bytearray((np.cumsum(a, axis=0) & 255).astype(np.uint8).reshape(-1)[:n].tobytes())
        elif ft == 2:
            cur = bytearray(((np.frombuffer(f, np.uint8).astype(np.int32) + np.frombuffer(bytes(prev), np.uint8))
                             & 255).astype(np.uint8).tobytes())
        else:
            cur = bytearray(n)
            for i in range(n):
                a = cur[i - unit] if i >= unit else 0
                b = prev[i]
                if ft == 3:
                    pred = (a + b) >> 1
                else:
                    c = prev[i - unit] if i >= unit else 0
                    pa, pb, pc = abs(b - c), abs(a - c), abs(a + b - 2 * c)
                    pred = a if pa <= pb and pa <= pc else (b if pb <= pc else c)
                cur[i] = (f[i] + pred) & 255
        out[r] = np.frombuffer(bytes(cur), np.uint8)
        prev = cur
    return out


def to_rgb(samples, colour, depth, palette=None) -> np.ndarray:
    """samples [h, w, ch] -> uint8 RGB [h, w, 3] under the decode contract (module docstring)"""
    s = samples.astype(np.uint32)
    if colour == 3:
        pal = np.zeros((256, 3), np.uint8)
        p = np.frombuffer(bytes(palette), np.uint8).reshape(-1, 3)
        pal[:len(p)] = p
        return pal[s[..., 0]]
    if depth == 16:
        s = s >> 8
    elif depth < 8:
        s = s * {1: 255, 2: 85, 4: 17}[depth]
    if colour in (0, 4):
        return np.repeat(s[..., :1], 3, axis=2).astype(np.uint8)
    return s[..., :3].astype(np.uint8)


def random_samples(px, colour, depth, seed=0, npal=None) -> np.ndarray:
    """[px, px, ch] samples: a smooth gradient plus noise (so every filter predicts something), full range for depth;
    palette indices run over all 2^depth values (past npal too when npal is smaller)"""
    rng = np.random.default_rng(seed)
    ch = CHANNELS[colour]
    top = (1 << depth) - 1
    y, x = np.mgrid[0:px, 0:px]
    base = ((x[..., None] * 3 + y[..., None] * 5 + np.arange(ch) * 17) * max(1, top // 64)) % (top + 1)
    noise = rng.integers(-(top // 16) - 1, top // 16 + 2, (px, px, ch))
    s = (base + noise) % (top + 1)
    if colour == 3:
        s = rng.integers(0, top + 1, (px, px, 1))
    return s.astype(np.uint16)


def random_palette(n, seed=0) -> bytes:
    return np.random.default_rng(seed + 1000).integers(0, 256, (n, 3), dtype=np.uint8).tobytes()


def filtered(samples, colour, depth, interlace=0, filters="random", seed=0) -> bytes:
    """the decompressed stream of `samples` [h, w, ch]: every non-empty pass's rows, each with its filter byte;
    filters = one type 0-4 for every row of every pass, or "random" (a random type per row)"""
    h, w, _ = samples.shape
    rng = np.random.default_rng(seed)
    raw = bytearray()
    for _, x0, y0, dx, dy, pw, ph in passes(w, h, interlace):
        sub = samples[y0::dy, x0::dx]
        ft = rng.integers(0, 5, ph) if filters == "random" else [filters] * ph
        raw += filter_rows(pack(sub, depth), ft, bpp(colour, depth))
    return bytes(raw)


def assemble(w, h, colour, depth, interlace, z: bytes, palette=None, trns=None, idat_size=None, before=()) -> bytes:
    """PNG file around the zlib stream z: palette = PLTE payload, trns = tRNS payload, before = chunks before PLTE"""
    step = idat_size or max(1, len(z))
    out = SIGNATURE + ihdr(w, h, depth, colour, interlace) + b"".join(before)
    if palette is not None:
        out += chunk(b"PLTE", palette)
    if trns is not None:
        out += chunk(b"tRNS", trns)
    out += b"".join(chunk(b"IDAT", z[i:i + step]) for i in range(0, len(z), step))
    return out + chunk(b"IEND", b"")


def encode(samples, colour, depth, interlace=0, filters="random", palette=None, seed=0, level=6, trns=None,
           idat_size=None, before=()) -> bytes:
    """PNG file of `samples` [h, w, ch] (see `filtered` and `assemble`)"""
    h, w, _ = samples.shape
    z = zlib.compress(filtered(samples, colour, depth, interlace, filters, seed), level)
    return assemble(w, h, colour, depth, interlace, z, palette, trns, idat_size, before)


def make(px, colour, depth, interlace=0, filters="random", seed=0, npal=None, **kw):
    """(file bytes, expected RGB8) of a synthetic tile; palette images get `npal` entries (default 2^depth - 1 capped
    at 256, so the top index is out of range and decodes black)"""
    s = random_samples(px, colour, depth, seed)
    pal = None
    if colour == 3:
        pal = random_palette(npal or min(256, max(1, (1 << depth) - 1)), seed)
    b = encode(s, colour, depth, interlace, filters, pal, seed, **kw)
    return b, to_rgb(s, colour, depth, pal)


def read_chunks(b: bytes):
    assert b[:8] == SIGNATURE
    i, out = 8, []
    while i < len(b):
        (n,) = struct.unpack(">I", b[i:i + 4])
        out.append((b[i + 4:i + 8], b[i + 8:i + 8 + n]))
        i += 12 + n
    return out


def decode(b: bytes) -> np.ndarray:
    """the reference decode of a PNG file to uint8 RGB [h, w, 3]"""
    chunks = read_chunks(b)
    w, h, depth, colour, _, _, interlace = struct.unpack(">IIBBBBB", chunks[0][1])
    palette = b"".join(d for t, d in chunks if t == b"PLTE") if colour == 3 else None
    data = zlib.decompress(b"".join(d for t, d in chunks if t == b"IDAT"))
    ch = CHANNELS[colour]
    samples = np.zeros((h, w, ch), np.uint16)
    pos = 0
    for _, x0, y0, dx, dy, pw, ph in passes(w, h, interlace):
        n = row_bytes(pw, colour, depth) - 1
        rows = unfilter(data[pos:pos + ph * (n + 1)], ph, n, bpp(colour, depth))
        samples[y0::dy, x0::dx] = unpack(rows, pw, ch, depth)
        pos += ph * (n + 1)
    if pos != len(data):
        raise ValueError(f"decompressed {len(data)} bytes, IHDR implies {pos}")
    return to_rgb(samples, colour, depth, palette)


def stream_size(px, colour, depth, interlace) -> int:
    return sum(ph * row_bytes(pw, colour, depth) for _, _, _, _, _, pw, ph in passes(px, px, interlace))


def first_mismatch(got, want, tile_labels, meta):
    """None, or a report of the first differing tiles as (tile, pass, row in the pass, column in the pass);
    meta[t] = (width, interlace)"""
    bad = np.flatnonzero((got != want).reshape(len(got), -1).any(1))
    if not bad.size:
        return None
    lines = [f"{bad.size} of {len(got)} tiles differ"]
    for t in bad[:5]:
        yx = np.argwhere((got[t] != want[t]).any(-1))
        y, x = (int(v) for v in yx[0])
        w, interlace = meta[t]
        where = f"row {y} column {x}"
        for p, x0, y0, dx, dy, _, _ in passes(w, w, interlace):
            if (x - x0) % dx == 0 and (y - y0) % dy == 0 and x >= x0 and y >= y0:
                where = f"pass {p + 1} row {(y - y0) // dy} column {(x - x0) // dx} (image row {y} column {x})"
                break
        lines.append(f"  tile {t} ({tile_labels[t]}): {len(yx)} pixels differ; first at {where}: got "
                     f"{got[t][y, x]} want {want[t][y, x]}")
    return "\n".join(lines)
