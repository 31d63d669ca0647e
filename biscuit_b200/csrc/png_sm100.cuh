// PNG decode kernels (sm_100a).  Included by png.cu only.  Three launches per group of tiles:
//   (a) png_dechunk_kernel   one CTA per tile: walks the run of IDAT chunks and copies their payloads into one
//                            contiguous zlib stream;
//   (b) png_inflate_kernel   one warp per tile: DEFLATE (RFC 1951) with zlib's validity rules.  Lane 0 decodes the
//                            Huffman symbols and writes literals; the warp copies each match;
//   (c) png_unfilter_kernel  one warp per tile, 8-bit RGB non-interlaced tiles (the default decode): reverses the five
//                            PNG filters over a diagonal wavefront of 32 rows, checks the Adler-32 of the decompressed
//                            stream, writes NHWC uint8;
//       png_unfilter_any_kernel  the same for every colour type, bit depth and interlace (BQ_PNG_CONVERT_RGB), pass by
//                            pass, converting each unfiltered row group to RGB8 before it writes it.
#pragma once

#include <stdint.h>

namespace bq {
namespace png {

// Per-tile descriptor built by the host chunk parse (png.cu).  Offsets are relative to the group it belongs to.
struct Tile {
  int64_t off;     // tile bytes = [off, off + len) of the group's byte buffer; its zlib stream goes to the same offset
  int32_t len;
  int32_t idat;    // first IDAT chunk (its length field), relative to the tile start
  int64_t foff;    // its decompressed (filtered) stream = [foff, foff + raw) of the group's filtered scratch
  int32_t raw;     // size of that stream, as IHDR implies
  uint8_t colour, depth, interlace;
  uint8_t bpp;     // bytes per filter unit: max(1, channels x depth / 8)
  int32_t npal;    // PLTE entries (palette images); pal holds them, zero-filled to 256
  uint8_t pal[768];
};

__device__ __forceinline__ uint32_t be32(const uint8_t* p) {
  return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | (uint32_t)p[3];
}

// ------------------------------------------------------------------------------------------------------------------
// (a) IDAT run -> zlib stream.  Thread 0 walks up to kSegs chunk headers, then the block copies their payloads.  IDAT
// CRCs are not checked (as in Pillow); the Adler-32 covers the data.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kDechunkThreads = 256, kSegs = 128;

__global__ void __launch_bounds__(kDechunkThreads) png_dechunk_kernel(const Tile* __restrict__ tiles,
                                                                       const uint8_t* __restrict__ data,
                                                                       uint8_t* __restrict__ zbuf,
                                                                       int32_t* __restrict__ zlen,
                                                                       int32_t* __restrict__ status) {
  __shared__ int32_t s_src[kSegs], s_dst[kSegs], s_len[kSegs];
  __shared__ int s_n, s_done, s_total;
  const Tile t = tiles[blockIdx.x];
  const uint8_t* src = data + t.off;
  uint8_t* dst = zbuf + t.off;
  int64_t p = t.idat;      // thread 0: next chunk header
  int32_t total = 0;
  for (;;) {
    if (threadIdx.x == 0) {
      int k = 0, done = 0;
      while (k < kSegs) {
        if (p + 8 > t.len || src[p + 4] != 'I' || src[p + 5] != 'D' || src[p + 6] != 'A' || src[p + 7] != 'T') {
          done = 1;        // the run ends at the next chunk of another type, or at the end of the file
          break;
        }
        const int64_t L = be32(src + p);
        if (L > (int64_t)t.len - p - 12) { done = 2; break; }   // the chunk runs past the tile's bytes
        s_src[k] = (int32_t)(p + 8);
        s_dst[k] = total;
        s_len[k] = (int32_t)L;
        total += (int32_t)L;
        ++k;
        p += 12 + L;
      }
      s_n = k;
      s_done = done;
      s_total = total;
    }
    __syncthreads();
    const int n = s_n, done = s_done;
    for (int k = 0; k < n; ++k) {
      const uint8_t* a = src + s_src[k];
      uint8_t* b = dst + s_dst[k];
      for (int i = threadIdx.x; i < s_len[k]; i += kDechunkThreads) b[i] = a[i];
    }
    __syncthreads();
    if (done) break;
  }
  if (threadIdx.x == 0) {
    zlen[blockIdx.x] = s_total;
    if (s_done == 2 || s_total < 2) status[blockIdx.x] = BQ_PNG_TRUNCATED_DATA;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// (b) inflate
// ------------------------------------------------------------------------------------------------------------------
constexpr int kInflateWarps = 4;
constexpr int kRoot = 10;              // bits of the primary lookup table; longer codes take the canonical slow path

// table entry: bits 0-3 code length (0: not in the primary table), 4-7 extra bits, 8-9 kind, 16-31 value
enum { kLit = 0, kLenDist = 1, kEob = 2, kInvalid = 3 };

__constant__ uint16_t kLenBase[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23, 27,
                                      31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t kDistBase[30] = {1,   2,   3,   4,   5,   7,    9,    13,   17,   25,   33,   49,   65,    97,    129,
                                       193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t kDistExtra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t kClOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct Huff {
  uint16_t count[16];    // codes of each length
  uint16_t sym[288];     // symbols in canonical order
};

struct Tables {
  uint32_t lit[1 << kRoot], dist[1 << kRoot];
  Huff hl, hd;           // hd doubles as the code-length code while a dynamic header is read
  uint8_t lens[320];
};

__device__ __forceinline__ uint32_t make_entry(int sym, bool dist, int len) {
  if (dist) {
    if (sym < 30) return len | kDistExtra[sym] << 4 | kLenDist << 8 | (uint32_t)kDistBase[sym] << 16;
    return len | kInvalid << 8;                       // distance codes 30 / 31 of the fixed code
  }
  if (sym < 256) return len | kLit << 8 | (uint32_t)sym << 16;
  if (sym == 256) return len | kEob << 8;
  if (sym < 286) return len | kLenExtra[sym - 257] << 4 | kLenDist << 8 | (uint32_t)kLenBase[sym - 257] << 16;
  return len | kInvalid << 8;                         // literal/length symbols 286 / 287 of the fixed code
}

// puff.c's canonical decode of the first `maxlen` bits (LSB first): the symbol, or -1 when no code matches
__device__ __forceinline__ int canon(uint32_t bits, int maxlen, const Huff& h, int& len) {
  int code = 0, first = 0, index = 0;
  for (int l = 1; l <= maxlen; ++l) {
    code |= (bits >> (l - 1)) & 1;
    const int c = h.count[l];
    if (code < first + c) { len = l; return h.sym[index + code - first]; }
    index += c;
    first = (first + c) << 1;
    code <<= 1;
  }
  return -1;
}

// Count / sort the code lengths (one lane).  zlib's inflate_table rules: an over-subscribed set is an error; an
// incomplete one too, except a single code of length 1 -- and no codes at all, which only fails when a symbol is
// decoded.  `codes` (the code-length code) allows neither.
__device__ bool huff_init(Huff& h, const uint8_t* lens, int n, bool codes) {
  for (int l = 0; l < 16; ++l) h.count[l] = 0;
  for (int s = 0; s < n; ++s) ++h.count[lens[s]];
  int left = 1, max = 0;
  for (int l = 1; l < 16; ++l) {
    left = (left << 1) - h.count[l];
    if (left < 0) return false;
    if (h.count[l]) max = l;
  }
  if (max == 0) { if (codes) return false; }
  else if (left > 0 && (codes || max != 1)) return false;
  uint16_t offs[16];
  offs[1] = 0;
  for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + h.count[l];
  for (int s = 0; s < n; ++s)
    if (lens[s]) h.sym[offs[lens[s]]++] = (uint16_t)s;
  h.count[0] = 0;
  return true;
}

// the primary table, one entry per kRoot-bit pattern, filled by the warp
__device__ __forceinline__ void fill_table(uint32_t* tab, const Huff& h, bool dist, int lane) {
  for (int i = lane; i < (1 << kRoot); i += 32) {
    int len = 0;
    const int s = canon((uint32_t)i, kRoot, h, len);
    tab[i] = s < 0 ? 0u : make_entry(s, dist, len);
  }
}

// LSB-first bit reader of lane 0 over stream bytes [0, end).  Bytes past the end read as 0; `pos` counts every byte
// loaded, so the stream was overrun when more bits were consumed than it holds.
struct Bits {
  const uint8_t* p;
  int64_t pos, end;
  uint64_t buf;
  int nb;
  __device__ __forceinline__ void refill() {
    if (nb <= 32) {
      uint32_t w;
      if (pos + 4 <= end) {
        w = (uint32_t)p[pos] | (uint32_t)p[pos + 1] << 8 | (uint32_t)p[pos + 2] << 16 | (uint32_t)p[pos + 3] << 24;
      } else {
        w = 0;
        for (int k = 0; k < 4; ++k)
          if (pos + k < end) w |= (uint32_t)p[pos + k] << (8 * k);
      }
      buf |= (uint64_t)w << nb;
      nb += 32;
      pos += 4;
    }
  }
  __device__ __forceinline__ uint32_t get(int n) {    // n <= 32, after refill() when n > nb
    const uint32_t v = (uint32_t)buf & ((1u << n) - 1u);
    buf >>= n;
    nb -= n;
    return v;
  }
  __device__ __forceinline__ void drop(int n) { buf >>= n; nb -= n; }
  __device__ __forceinline__ int64_t consumed_bits() const { return pos * 8 - nb; }
  __device__ __forceinline__ bool overrun() const { return consumed_bits() > end * 8; }
};

enum { kCtlMatch = 1, kCtlEob = 2 };

// Tile `tile` of the group: zlib stream zbuf[off, off + zlen) (the 2-byte header was checked on the host) ->
// filt[foff, foff + raw), its Adler-32 trailer -> adler[tile].
__global__ void __launch_bounds__(32 * kInflateWarps) png_inflate_kernel(const Tile* __restrict__ tiles,
                                                                          const uint8_t* __restrict__ zbuf,
                                                                          const int32_t* __restrict__ zlen, int n_tiles,
                                                                          uint8_t* __restrict__ filt,
                                                                          uint32_t* __restrict__ adler,
                                                                          int32_t* __restrict__ status) {
  __shared__ Tables tabs[kInflateWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x * kInflateWarps + warp;
  if (tile >= n_tiles || status[tile] != 0) return;   // whole warps leave together
  Tables& T = tabs[warp];
  const int32_t raw = tiles[tile].raw;
  uint8_t* out = filt + tiles[tile].foff;
  Bits br;
  br.p = zbuf + tiles[tile].off + 2;
  br.end = zlen[tile] - 2;
  br.pos = 0;
  br.buf = 0;
  br.nb = 0;
  int err = 0, loaded = 0;      // loaded: 1 = the fixed code is in T, 2 = a dynamic code
  int32_t opos = 0;             // lane 0: bytes written
  bool final = false;
  while (!final) {
    int btype = 0, nlit = 0, ndist = 0;
    if (lane == 0) {
      br.refill();
      final = br.get(1);
      btype = (int)br.get(2);
      if (btype == 3) {
        err = BQ_PNG_BAD_BLOCK;
      } else if (btype == 1) {
        nlit = 288;
        ndist = 32;
        if (loaded != 1) {
          for (int s = 0; s < 288; ++s) T.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
          for (int s = 0; s < 32; ++s) T.lens[288 + s] = 5;
        }
      } else if (btype == 2) {
        br.refill();
        nlit = (int)br.get(5) + 257;
        ndist = (int)br.get(5) + 1;
        const int ncl = (int)br.get(4) + 4;
        if (nlit > 286 || ndist > 30) err = BQ_PNG_BAD_HUFFMAN;
        uint8_t cl[19];
        for (int k = 0; k < 19; ++k) cl[k] = 0;
        for (int k = 0; k < ncl; ++k) { br.refill(); cl[kClOrder[k]] = (uint8_t)br.get(3); }
        if (!err && !huff_init(T.hd, cl, 19, true)) err = BQ_PNG_BAD_HUFFMAN;
        for (int k = 0; !err && k < nlit + ndist;) {
          br.refill();
          int len = 0;
          const int sym = canon((uint32_t)br.buf, 7, T.hd, len);
          if (sym < 0) { err = BQ_PNG_BAD_HUFFMAN; break; }
          br.drop(len);
          if (sym < 16) { T.lens[k++] = (uint8_t)sym; continue; }
          int rep, val = 0;
          if (sym == 16) {
            if (k == 0) { err = BQ_PNG_BAD_HUFFMAN; break; }     // repeat with no previous length
            val = T.lens[k - 1];
            rep = 3 + (int)br.get(2);
          } else if (sym == 17) {
            rep = 3 + (int)br.get(3);
          } else {
            rep = 11 + (int)br.get(7);
          }
          if (k + rep > nlit + ndist) { err = BQ_PNG_BAD_HUFFMAN; break; }
          while (rep--) T.lens[k++] = (uint8_t)val;
        }
        if (!err && T.lens[256] == 0) err = BQ_PNG_BAD_HUFFMAN;   // no end-of-block code
        // the fixed layout keeps its distance lengths at 288; a dynamic code's start right after its literal lengths
      }
      if (!err && btype != 0 && (btype == 2 || loaded != 1)) {
        const uint8_t* dl = T.lens + (btype == 1 ? 288 : nlit);
        if (!huff_init(T.hl, T.lens, nlit, false) || !huff_init(T.hd, dl, ndist, false)) err = BQ_PNG_BAD_HUFFMAN;
      }
      if (err && br.overrun()) err = BQ_PNG_TRUNCATED_DATA;
    }
    btype = __shfl_sync(0xFFFFFFFFu, btype, 0);
    err = __shfl_sync(0xFFFFFFFFu, err, 0);
    if (err) break;
    if (btype == 0) {
      // stored block: byte-align, LEN / NLEN, then LEN bytes copied by the warp
      int64_t src = 0;
      int32_t L = 0;
      if (lane == 0) {
        br.drop(br.nb & 7);
        br.refill();
        L = (int32_t)br.get(16);
        const int32_t nl = (int32_t)br.get(16);
        src = br.pos - br.nb / 8;
        if (br.overrun() || src + L > br.end) err = BQ_PNG_TRUNCATED_DATA;
        else if ((L ^ 0xFFFF) != nl) err = BQ_PNG_BAD_BLOCK;
        else if (opos + L > raw) err = BQ_PNG_WRONG_SIZE;
        br.pos = src + L;
        br.buf = 0;
        br.nb = 0;
      }
      err = __shfl_sync(0xFFFFFFFFu, err, 0);
      if (err) break;
      src = __shfl_sync(0xFFFFFFFFu, src, 0);
      L = __shfl_sync(0xFFFFFFFFu, L, 0);
      const int32_t o = __shfl_sync(0xFFFFFFFFu, opos, 0);
      for (int32_t i = lane; i < L; i += 32) out[o + i] = br.p[src + i];
      if (lane == 0) opos += L;
      __syncwarp();
    } else {
      if (btype == 2 || loaded != 1) {
        __syncwarp();
        fill_table(T.lit, T.hl, false, lane);
        fill_table(T.dist, T.hd, true, lane);
        loaded = btype;
        __syncwarp();
      }
      for (;;) {
        int ctl = 0, mlen = 0, mdist = 0;
        if (lane == 0) {
          for (;;) {
            br.refill();
            if (br.pos > br.end + 8) { err = BQ_PNG_TRUNCATED_DATA; break; }
            uint32_t e = T.lit[br.buf & ((1u << kRoot) - 1)];
            if ((e & 15) == 0) {
              int len = 0;
              const int s = canon((uint32_t)br.buf, 15, T.hl, len);
              if (s < 0) { err = BQ_PNG_BAD_HUFFMAN; break; }
              e = make_entry(s, false, len);
            }
            br.drop(e & 15);
            const uint32_t kind = (e >> 8) & 3;
            if (kind == kLit) {
              if (opos >= raw) { err = BQ_PNG_WRONG_SIZE; break; }
              out[opos++] = (uint8_t)(e >> 16);
              continue;
            }
            if (kind == kEob) { ctl = kCtlEob; break; }
            if (kind == kInvalid) { err = BQ_PNG_BAD_HUFFMAN; break; }
            mlen = (int)(e >> 16) + (int)br.get((e >> 4) & 15);
            br.refill();
            uint32_t d = T.dist[br.buf & ((1u << kRoot) - 1)];
            if ((d & 15) == 0) {
              int len = 0;
              const int s = canon((uint32_t)br.buf, 15, T.hd, len);
              if (s < 0) { err = BQ_PNG_BAD_HUFFMAN; break; }
              d = make_entry(s, true, len);
            }
            br.drop(d & 15);
            if (((d >> 8) & 3) == kInvalid) { err = BQ_PNG_BAD_HUFFMAN; break; }
            mdist = (int)(d >> 16) + (int)br.get((d >> 4) & 15);
            if (mdist > opos) { err = BQ_PNG_BAD_DISTANCE; break; }        // reaches before the start of the stream
            if (opos + mlen > raw) { err = BQ_PNG_WRONG_SIZE; break; }
            ctl = kCtlMatch;
            break;
          }
          if (err && br.overrun()) err = BQ_PNG_TRUNCATED_DATA;
        }
        __syncwarp();                                  // lane 0's literals are visible to the copy below
        ctl = __shfl_sync(0xFFFFFFFFu, ctl, 0);
        err = __shfl_sync(0xFFFFFFFFu, err, 0);
        if (ctl != kCtlMatch || err) break;
        mlen = __shfl_sync(0xFFFFFFFFu, mlen, 0);
        mdist = __shfl_sync(0xFFFFFFFFu, mdist, 0);
        const int32_t o = __shfl_sync(0xFFFFFFFFu, opos, 0);
        // out[o + i] = out[o - d + (i mod d)]: every source lies before o, so the copy has no rounds even when d < len
        for (int i = lane; i < mlen; i += 32) out[o + i] = out[o - mdist + (i < mdist ? i : i % mdist)];
        if (lane == 0) opos += mlen;
        __syncwarp();
      }
      if (err) break;
    }
    final = __shfl_sync(0xFFFFFFFFu, (int)final, 0);
  }
  if (lane == 0) {
    if (!err) {
      br.drop(br.nb & 7);                             // the Adler-32 follows the final block, byte-aligned, big-endian
      br.refill();
      uint32_t a = 0;
      for (int k = 0; k < 4; ++k) a = a << 8 | br.get(8);
      if (br.overrun()) err = BQ_PNG_TRUNCATED_DATA;
      else if (opos != raw) err = BQ_PNG_WRONG_SIZE;
      adler[tile] = a;
    }
    if (err) status[tile] = err;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// (c) unfilter.  One warp per tile owns 32 consecutive rows at a time, staged through shared memory.  At step s lane j
// reconstructs pixel x = s - j of row r0 + j: the pixel above comes from lane j - 1 (which finished it at step s - 1),
// the one above-left from the previous step, the left one from the lane's own previous step.  Every byte also enters
// the Adler-32 sums (sum b and sum (N - i) b, reduced mod 65521 at the end).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kRows = 32;

__host__ __device__ constexpr size_t unfilter_smem(int px) { return (size_t)(kRows + 1) * (1 + 3 * px); }

__device__ __forceinline__ uint32_t unfilter_px(int ft, uint32_t f, uint32_t a, uint32_t b, uint32_t c) {
  uint32_t v = 0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int fa = (a >> (8 * k)) & 255, fb = (b >> (8 * k)) & 255, fc = (c >> (8 * k)) & 255;
    int pred = 0;
    if (ft == 1) pred = fa;
    else if (ft == 2) pred = fb;
    else if (ft == 3) pred = (fa + fb) >> 1;
    else if (ft == 4) {
      const int pa = abs(fb - fc), pb = abs(fa - fc), pc = abs(fa + fb - 2 * fc);
      pred = (pa <= pb && pa <= pc) ? fa : (pb <= pc ? fb : fc);
    }
    v |= (uint32_t)((((f >> (8 * k)) & 255) + pred) & 255) << (8 * k);
  }
  return v;
}

__global__ void __launch_bounds__(32) png_unfilter_kernel(const uint8_t* __restrict__ filt, int px,
                                                          const uint32_t* __restrict__ adler,
                                                          int32_t* __restrict__ status, uint8_t* __restrict__ out) {
  extern __shared__ uint8_t sm[];
  const int tile = blockIdx.x, lane = threadIdx.x;
  if (status[tile] != 0) return;
  const int rowb = 1 + 3 * px;
  const int64_t raw = (int64_t)px * rowb;
  const uint8_t* f = filt + (size_t)tile * raw;
  uint8_t* o = out + (size_t)tile * px * px * 3;
  uint8_t* rows = sm;                                  // [kRows][rowb], unfiltered in place
  uint8_t* prev = sm + (size_t)kRows * rowb;           // the row above the group (zeros above row 0), same layout
  for (int i = lane; i < rowb; i += 32) prev[i] = 0;
  uint64_t sa = 0, sb = 0;
  int bad = 0;
  for (int r0 = 0; r0 < px; r0 += kRows) {
    const int nr = min(kRows, px - r0);
    const int64_t base = (int64_t)r0 * rowb;
    const int n = nr * rowb;
    for (int i = lane; i < n; i += 32) {
      const uint32_t b = f[base + i];
      rows[i] = (uint8_t)b;
      sa += b;
      sb += (uint64_t)(raw - base - i) * b;
    }
    __syncwarp();
    uint8_t* my = rows + (size_t)lane * rowb;
    int ft = lane < nr ? my[0] : 0;
    if (ft > 4) { bad = 1; ft = 0; }
    uint32_t cur = 0, upl = 0;                          // own previous pixel; the up value of the previous step
    for (int s = 0; s < px + nr - 1; ++s) {
      const int x = s - lane;
      uint32_t up = __shfl_up_sync(0xFFFFFFFFu, cur, 1);
      if (lane == 0 && x < px) up = prev[1 + 3 * x] | prev[2 + 3 * x] << 8 | prev[3 + 3 * x] << 16;
      if (x >= 0 && x < px && lane < nr) {
        uint8_t* q = my + 1 + 3 * x;
        const uint32_t fv = q[0] | q[1] << 8 | q[2] << 16;
        const uint32_t a = x ? cur : 0, c = x ? upl : 0;
        cur = unfilter_px(ft, fv, a, up, c);
        q[0] = (uint8_t)cur;
        q[1] = (uint8_t)(cur >> 8);
        q[2] = (uint8_t)(cur >> 16);
      }
      upl = up;
    }
    __syncwarp();
    const int64_t ob = (int64_t)r0 * px * 3;
    const int rb = 3 * px;
    for (int i = lane; i < nr * rb; i += 32) {
      const int r = i / rb;
      o[ob + i] = rows[(size_t)r * rowb + 1 + (i - r * rb)];
    }
    for (int i = lane; i < rowb; i += 32) prev[i] = rows[(size_t)(nr - 1) * rowb + i];
    __syncwarp();
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    sa += __shfl_xor_sync(0xFFFFFFFFu, sa, d);
    sb += __shfl_xor_sync(0xFFFFFFFFu, sb, d);
  }
  bad = __any_sync(0xFFFFFFFFu, bad);
  if (lane == 0) {
    const uint32_t A = (uint32_t)((1 + sa) % 65521), B = (uint32_t)(((uint64_t)raw + sb) % 65521);
    if ((B << 16 | A) != adler[tile]) status[tile] = BQ_PNG_ADLER;
    else if (bad) status[tile] = BQ_PNG_BAD_FILTER;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// (c') unfilter + convert, any colour type / bit depth / interlace.  One warp per tile walks the Adam7 passes (one pass
// when not interlaced) in stream order.  Within a pass it runs the wavefront of (c) over groups of 32 rows, on filter
// units of bpp bytes (1 to 8, held in a uint64), with the pass's row length 1 + ceil(w x channels x depth / 8).  Once a
// group is unfiltered in shared memory the warp converts each of its pixels to RGB8 -- sub-byte samples unpacked and
// scaled (gray) or looked up (palette), 16-bit samples reduced to the high byte, gray replicated, alpha dropped -- and
// writes it to (y0 + r dy, x0 + c dx).  The Adler-32 runs over the whole stream in stream order, across passes.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kPalBytes = 768;

// Adam7 passes 1-7 (indices 0-6): first column / row and their steps; index 7 is the whole non-interlaced image
__constant__ uint8_t kAdam7[8][4] = {{0, 0, 8, 8}, {4, 0, 8, 8}, {0, 4, 4, 8}, {2, 0, 4, 4},
                                     {0, 2, 2, 4}, {1, 0, 2, 2}, {0, 1, 1, 2}, {0, 0, 1, 1}};

__host__ __device__ constexpr int png_channels(int colour) {
  return colour == 2 ? 3 : colour == 4 ? 2 : colour == 6 ? 4 : 1;
}

// filtered row bytes of a pass `w` pixels wide
__host__ __device__ constexpr int64_t row_bytes(int64_t w, int colour, int depth) {
  return 1 + (w * png_channels(colour) * depth + 7) / 8;
}

// shared memory of png_unfilter_any_kernel for rows of at most `row` bytes
__host__ __device__ constexpr size_t unfilter_any_smem(int64_t row) { return kPalBytes + (size_t)(kRows + 1) * row; }

__device__ __forceinline__ uint64_t unfilter_unit(int ft, int bpp, uint64_t f, uint64_t a, uint64_t b, uint64_t c) {
  uint64_t v = 0;
  for (int k = 0; k < bpp; ++k) {
    const int fa = (int)(a >> (8 * k)) & 255, fb = (int)(b >> (8 * k)) & 255, fc = (int)(c >> (8 * k)) & 255;
    int pred = 0;
    if (ft == 1) pred = fa;
    else if (ft == 2) pred = fb;
    else if (ft == 3) pred = (fa + fb) >> 1;
    else if (ft == 4) {
      const int pa = abs(fb - fc), pb = abs(fa - fc), pc = abs(fa + fb - 2 * fc);
      pred = (pa <= pb && pa <= pc) ? fa : (pb <= pc ? fb : fc);
    }
    v |= (uint64_t)((((int)(f >> (8 * k)) & 255) + pred) & 255) << (8 * k);
  }
  return v;
}

__device__ __forceinline__ uint64_t load_unit(const uint8_t* p, int bpp) {
  uint64_t v = 0;
  for (int k = 0; k < bpp; ++k) v |= (uint64_t)p[k] << (8 * k);
  return v;
}

__global__ void __launch_bounds__(32) png_unfilter_any_kernel(const Tile* __restrict__ tiles,
                                                              const uint8_t* __restrict__ filt, int px,
                                                              const uint32_t* __restrict__ adler,
                                                              int32_t* __restrict__ status, uint8_t* __restrict__ out) {
  extern __shared__ uint8_t sm[];
  const int tile = blockIdx.x, lane = threadIdx.x;
  if (status[tile] != 0) return;
  const Tile& t = tiles[tile];
  const int colour = t.colour, depth = t.depth, bpp = t.bpp, ch = png_channels(colour);
  const int64_t raw = t.raw;
  const uint8_t* f = filt + t.foff;
  uint8_t* o = out + (size_t)tile * px * px * 3;
  uint8_t* pal = sm;                                   // [256][3], zero past the PLTE entries
  uint8_t* rows = sm + kPalBytes;
  for (int i = lane; i < kPalBytes; i += 32) pal[i] = t.pal[i];
  const int gray_scale = depth == 1 ? 255 : depth == 2 ? 85 : depth == 4 ? 17 : 1;
  uint64_t sa = 0, sb = 0;
  int64_t pos = 0;                                     // stream offset of the pass
  int bad = 0;
  for (int p = t.interlace ? 0 : 7; p < (t.interlace ? 7 : 8); ++p) {
    const int x0 = kAdam7[p][0], y0 = kAdam7[p][1], dx = kAdam7[p][2], dy = kAdam7[p][3];
    const int pw = px > x0 ? (px - x0 + dx - 1) / dx : 0, ph = px > y0 ? (px - y0 + dy - 1) / dy : 0;
    if (pw == 0 || ph == 0) continue;                  // an empty pass has no bytes, not even filter bytes
    const int rowb = (int)row_bytes(pw, colour, depth);
    const int units = (rowb - 1) / bpp;                // sub-byte rows: one unit per byte
    uint8_t* prev = rows + (size_t)kRows * rowb;       // the row above the group (zeros above the pass's row 0)
    __syncwarp();
    for (int i = lane; i < rowb; i += 32) prev[i] = 0;
    for (int r0 = 0; r0 < ph; r0 += kRows) {
      const int nr = min(kRows, ph - r0);
      const int64_t base = pos + (int64_t)r0 * rowb;
      const int n = nr * rowb;
      for (int i = lane; i < n; i += 32) {
        const uint32_t b = f[base + i];
        rows[i] = (uint8_t)b;
        sa += b;
        sb += (uint64_t)(raw - base - i) * b;
      }
      __syncwarp();
      uint8_t* my = rows + (size_t)lane * rowb;
      int ft = lane < nr ? my[0] : 0;
      if (ft > 4) { bad = 1; ft = 0; }
      uint64_t cur = 0, upl = 0;                       // own previous unit; the up value of the previous step
      for (int s = 0; s < units + nr - 1; ++s) {
        const int x = s - lane;
        uint64_t up = __shfl_up_sync(0xFFFFFFFFu, cur, 1);
        if (lane == 0 && x >= 0 && x < units) up = load_unit(prev + 1 + bpp * x, bpp);
        if (x >= 0 && x < units && lane < nr) {
          uint8_t* q = my + 1 + bpp * x;
          const uint64_t a = x ? cur : 0, c = x ? upl : 0;
          cur = unfilter_unit(ft, bpp, load_unit(q, bpp), a, up, c);
          for (int k = 0; k < bpp; ++k) q[k] = (uint8_t)(cur >> (8 * k));
        }
        upl = up;
      }
      __syncwarp();
      for (int i = lane; i < nr * pw; i += 32) {
        const int r = i / pw, c = i - r * pw;
        const uint8_t* q = rows + (size_t)r * rowb + 1;
        uint32_t R, G, B;
        if (depth < 8) {
          const int bit = c * depth;
          const uint32_t v = (q[bit >> 3] >> (8 - depth - (bit & 7))) & ((1u << depth) - 1u);
          if (colour == 3) { R = pal[3 * v]; G = pal[3 * v + 1]; B = pal[3 * v + 2]; }
          else R = G = B = v * gray_scale;
        } else {
          const int sh = depth >> 4;                   // 16-bit samples: the high (first) byte
          const uint8_t* e = q + ((size_t)c * ch << sh);
          if (colour == 3) { R = pal[3 * e[0]]; G = pal[3 * e[0] + 1]; B = pal[3 * e[0] + 2]; }
          else if (colour == 0 || colour == 4) R = G = B = e[0];
          else { R = e[0]; G = e[1 << sh]; B = e[2 << sh]; }
        }
        uint8_t* d = o + ((size_t)(y0 + (r0 + r) * dy) * px + x0 + (size_t)c * dx) * 3;
        d[0] = (uint8_t)R;
        d[1] = (uint8_t)G;
        d[2] = (uint8_t)B;
      }
      for (int i = lane; i < rowb; i += 32) prev[i] = rows[(size_t)(nr - 1) * rowb + i];
      __syncwarp();
    }
    pos += (int64_t)ph * rowb;
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    sa += __shfl_xor_sync(0xFFFFFFFFu, sa, d);
    sb += __shfl_xor_sync(0xFFFFFFFFu, sb, d);
  }
  bad = __any_sync(0xFFFFFFFFu, bad);
  if (lane == 0) {
    const uint32_t A = (uint32_t)((1 + sa) % 65521), B = (uint32_t)(((uint64_t)raw + sb) % 65521);
    if ((B << 16 | A) != adler[tile]) status[tile] = BQ_PNG_ADLER;
    else if (bad) status[tile] = BQ_PNG_BAD_FILTER;
  }
}

}  // namespace png
}  // namespace bq
