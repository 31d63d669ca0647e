"""numpy restatement of libjpeg-turbo's default baseline decode (test oracle only).

The four stages the GPU decoder (biscuit_b200/csrc/jpeg_sm100.cuh) runs, written out plainly so a GPU mismatch can be
localised to one of them:

  1. marker parse + byte unstuffing + Huffman decode (jdhuff.c), DC prediction reset at every restart marker;
  2. dequantisation + JDCT_ISLOW integer IDCT (jidctint.c) with the post-IDCT range limit;
  3. fancy (triangular) upsampling of 4:2:2 / 4:2:0 chroma (jdsample.c h2v1 / h2v2, edge samples replicated);
  4. fixed-point YCbCr -> RGB (jdcolor.c), cropped to the image size.

`decode(b)` equals `np.asarray(PIL.Image.open(io.BytesIO(b)).convert("RGB"))` bit for bit on every encoding the GPU
decoder accepts (tests/test_jpeg_cpu.py pins it).  The Huffman stage is a plain Python loop: a few tiles per test.
"""
from __future__ import annotations

import numpy as np

ZIGZAG = np.array([
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55,
    62, 63])   # zig-zag index -> natural (row-major) index


def parse(b: bytes) -> dict:
    """Header fields of a baseline 3-component JPEG (no validation beyond what decoding needs)."""
    i, qt, ht, ri, comps, scan = 2, {}, {}, 0, None, None
    while True:
        while b[i] != 0xFF:
            i += 1
        while b[i] == 0xFF:
            i += 1
        m = b[i]
        i += 1
        ln = (b[i] << 8) | b[i + 1]
        seg = b[i + 2:i + ln]
        if m == 0xDB:
            k = 0
            while k < len(seg):
                pq, tq = seg[k] >> 4, seg[k] & 15
                n = 128 if pq else 64
                raw = np.frombuffer(seg[k + 1:k + 1 + n], ">u2" if pq else "u1").astype(np.int32)
                tab = np.zeros(64, np.int32)
                tab[ZIGZAG] = raw
                qt[tq] = tab
                k += 1 + n
        elif m == 0xC4:
            k = 0
            while k < len(seg):
                tc, th = seg[k] >> 4, seg[k] & 15
                bits = list(seg[k + 1:k + 17])
                vals = list(seg[k + 17:k + 17 + sum(bits)])
                ht[(tc, th)] = _huff_table(bits, vals)
                k += 17 + sum(bits)
        elif m == 0xDD:
            ri = (seg[0] << 8) | seg[1]
        elif m in (0xC0, 0xC1):
            h, w, nc = (seg[1] << 8) | seg[2], (seg[3] << 8) | seg[4], seg[5]
            comps = [dict(id=seg[6 + 3 * c], h=seg[7 + 3 * c] >> 4, v=seg[7 + 3 * c] & 15, tq=seg[8 + 3 * c])
                     for c in range(nc)]
        elif m == 0xDA:
            ns = seg[0]
            scan = [(seg[1 + 2 * c], seg[2 + 2 * c] >> 4, seg[2 + 2 * c] & 15) for c in range(ns)]
            start = i + ln
            break
        i += ln
    byid = {c["id"]: c for c in comps}
    for cid, td, ta in scan:
        byid[cid]["td"], byid[cid]["ta"] = td, ta
    return dict(height=h, width=w, comps=comps, qt=qt, ht=ht, restart=ri, scan_start=start)


def _huff_table(bits, vals):
    """code (as (length, value)) -> symbol, jdhuff.c's canonical code assignment"""
    table, code, k = {}, 0, 0
    for ln in range(1, 17):
        for _ in range(bits[ln - 1]):
            table[(ln, code)] = vals[k]
            code += 1
            k += 1
        code <<= 1
    return table


def _unstuff(data: bytes):
    """entropy-coded bytes without FF00 stuffing, split at RSTn markers; stops at the first other marker"""
    out, cur, i = [], bytearray(), 0
    while i < len(data):
        x = data[i]
        if x != 0xFF:
            cur.append(x)
            i += 1
            continue
        nx = data[i + 1]
        if nx == 0x00:
            cur.append(0xFF)
            i += 2
        elif nx == 0xFF:
            i += 1
        elif 0xD0 <= nx <= 0xD7:
            out.append(bytes(cur))
            cur = bytearray()
            i += 2
        else:
            break
    out.append(bytes(cur))
    return out


class _Bits:
    def __init__(self, data: bytes):
        self.v = int.from_bytes(data, "big") if data else 0
        self.n = 8 * len(data)
        self.p = 0

    def get(self, k):
        if k == 0:
            return 0
        if self.p + k > self.n:
            raise ValueError("entropy segment ran out of bits")
        x = (self.v >> (self.n - self.p - k)) & ((1 << k) - 1)
        self.p += k
        return x

    def symbol(self, table):
        code = 0
        for ln in range(1, 17):
            code = (code << 1) | self.get(1)
            s = table.get((ln, code))
            if s is not None:
                return s
        raise ValueError("invalid Huffman code")


def _extend(x, s):
    return x - (1 << s) + 1 if s and x < (1 << (s - 1)) else x


def coefficients(hdr: dict, b: bytes):
    """per component: dequantised-ready int coefficient blocks [by, bx, 64] in natural order (DC already predicted)"""
    comps = hdr["comps"]
    hmax, vmax = max(c["h"] for c in comps), max(c["v"] for c in comps)
    mcux = -(-hdr["width"] // (8 * hmax))
    mcuy = -(-hdr["height"] // (8 * vmax))
    out = [np.zeros((mcuy * c["v"], mcux * c["h"], 64), np.int32) for c in comps]
    intervals = _unstuff(b[hdr["scan_start"]:])
    ri = hdr["restart"] or mcux * mcuy
    mcu = 0
    for seg in intervals:
        if mcu >= mcux * mcuy:
            break
        bits, pred = _Bits(seg), [0] * len(comps)
        for _ in range(min(ri, mcux * mcuy - mcu)):
            my, mx = divmod(mcu, mcux)
            for ci, c in enumerate(comps):
                dc, ac = hdr["ht"][(0, c["td"])], hdr["ht"][(1, c["ta"])]
                for dy in range(c["v"]):
                    for dx in range(c["h"]):
                        blk = out[ci][my * c["v"] + dy, mx * c["h"] + dx]
                        s = bits.symbol(dc)
                        pred[ci] += _extend(bits.get(s), s)
                        blk[0] = pred[ci]
                        k = 1
                        while k < 64:
                            rs = bits.symbol(ac)
                            r, s = rs >> 4, rs & 15
                            if s == 0:
                                if r != 15:
                                    break
                                k += 16
                                continue
                            k += r
                            if k > 63:
                                raise ValueError("AC run past the end of the block")
                            blk[ZIGZAG[k]] = _extend(bits.get(s), s)
                            k += 1
            mcu += 1
    return out, (mcux, mcuy, hmax, vmax)


def idct_islow(coef: np.ndarray, q: np.ndarray) -> np.ndarray:
    """jidctint.c jpeg_idct_islow on blocks [..., 64] (natural order) -> uint8 [..., 8, 8].  Every step is exact
    integer arithmetic; the final range limit is libjpeg-turbo's SIMD one (saturate to [0, 255] after +128), which
    equals the C table lookup for every |value| < 512."""
    x = (coef.astype(np.int64) * q.astype(np.int64)).reshape(coef.shape[:-1] + (8, 8))

    def one_pass(v, shift):           # v[..., 8 (along the transform), m]
        z2, z3 = v[..., 2, :], v[..., 6, :]
        z1 = (z2 + z3) * 4433
        tmp2 = z1 + z3 * -15137
        tmp3 = z1 + z2 * 6270
        tmp0 = (v[..., 0, :] + v[..., 4, :]) << 13
        tmp1 = (v[..., 0, :] - v[..., 4, :]) << 13
        t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
        o0, o1, o2, o3 = v[..., 7, :], v[..., 5, :], v[..., 3, :], v[..., 1, :]
        z1, z2, z3, z4 = o0 + o3, o1 + o2, o0 + o2, o1 + o3
        z5 = (z3 + z4) * 9633
        o0, o1, o2, o3 = o0 * 2446, o1 * 16819, o2 * 25172, o3 * 12299
        z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
        o0, o1, o2, o3 = o0 + z1 + z3, o1 + z2 + z4, o2 + z2 + z3, o3 + z1 + z4
        r = 1 << (shift - 1)
        outs = [t10 + o3, t11 + o2, t12 + o1, t13 + o0, t13 - o0, t12 - o1, t11 - o2, t10 - o3]
        return np.stack([(o + r) >> shift for o in outs], axis=-2)

    ws = one_pass(x, 11)                                          # columns: transform along rows index
    ws = np.swapaxes(one_pass(np.swapaxes(ws, -1, -2), 18), -1, -2)
    return np.clip(ws + 128, 0, 255).astype(np.uint8)


def planes(hdr, coef):
    out = []
    for c, blocks in zip(hdr["comps"], coef):
        px = idct_islow(blocks, hdr["qt"][c["tq"]])               # [by, bx, 8, 8]
        by, bx = px.shape[:2]
        out.append(px.transpose(0, 2, 1, 3).reshape(by * 8, bx * 8))
    return out


def _fancy_h2v1(p):
    """jdsample.c h2v1_fancy_upsample on a [H, W] plane (W = downsampled width)"""
    p = p.astype(np.int32)
    left = np.concatenate([p[:, :1], p[:, :-1]], 1)
    right = np.concatenate([p[:, 1:], p[:, -1:]], 1)
    out = np.empty((p.shape[0], 2 * p.shape[1]), np.int32)
    out[:, 0::2] = (3 * p + left + 1) >> 2
    out[:, 1::2] = (3 * p + right + 2) >> 2
    return out


def _fancy_h2v2(p):
    """jdsample.c h2v2_fancy_upsample (rows above the first / below the last replicate the edge row)"""
    p = p.astype(np.int32)
    up = np.concatenate([p[:1], p[:-1]], 0)
    down = np.concatenate([p[1:], p[-1:]], 0)
    out = np.empty((2 * p.shape[0], 2 * p.shape[1]), np.int32)
    for v, far in ((0, up), (1, down)):
        cs = 3 * p + far
        left = np.concatenate([cs[:, :1], cs[:, :-1]], 1)
        right = np.concatenate([cs[:, 1:], cs[:, -1:]], 1)
        out[v::2, 0::2] = (3 * cs + left + 8) >> 4
        out[v::2, 1::2] = (3 * cs + right + 7) >> 4
    return out


def ycc_to_rgb(y, cb, cr):
    """jdcolor.c ycc_rgb_convert (SCALEBITS 16 tables, arithmetic right shifts)"""
    y, cb, cr = (a.astype(np.int64) for a in (y, cb, cr))
    half = 1 << 15
    xb, xr = cb - 128, cr - 128
    r = y + ((91881 * xr + half) >> 16)
    g = y + ((-46802 * xr + -22554 * xb + half) >> 16)
    b = y + ((116130 * xb + half) >> 16)
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)


def decode(b: bytes) -> np.ndarray:
    hdr = parse(b)
    coef, (mcux, mcuy, hmax, vmax) = coefficients(hdr, b)
    pl = planes(hdr, coef)
    H, W = hdr["height"], hdr["width"]
    full = [pl[0][:H, :W]]
    for c, p in zip(hdr["comps"][1:], pl[1:]):
        dh, dw = -(-H * c["v"] // vmax), -(-W * c["h"] // hmax)      # jdinput.c downsampled_height / _width
        p = p[:dh, :dw]
        if (hmax // c["h"], vmax // c["v"]) == (2, 2):
            p = _fancy_h2v2(p)
        elif (hmax // c["h"], vmax // c["v"]) == (2, 1):
            p = _fancy_h2v1(p)
        full.append(p[:H, :W])
    return ycc_to_rgb(*full)
