// Baseline-JPEG decode kernels (sm_100a), bit-exact with libjpeg-turbo's decompression (jdcolor.c tables) under the two
// options TensorFlow's decode_jpeg exposes: the IDCT (JDCT_ISLOW, libjpeg-turbo's default, or JDCT_IFAST) and fancy or
// replicated (merged) chroma upsampling.  Included by jpeg.cu only.  Four launches per batch of tiles, one CTA per tile
// for the first two:
//   (a) jpeg_unstuff_kernel   removes FF00 stuffing and RSTn markers, records where each restart interval starts;
//   (b) jpeg_huffman_kernel   parallel Huffman decode by self-synchronising subsequences (Weissenberger & Schmidt,
//                             ICPP 2018), then the DC prediction per component per restart interval;
//   (c) jpeg_idct_kernel      dequantisation + ISLOW or IFAST IDCT -> component planes;
//   (d) jpeg_color_kernel     fancy or replicated upsampling + YCbCr->RGB + crop, NHWC uint8 into the caller's tile
//                             buffer.
#pragma once

#include <cub/block/block_scan.cuh>
#include <stdint.h>

namespace bq {
namespace jpeg {

constexpr int kMaxBpm = 6;            // blocks per MCU of the accepted samplings (4:2:0 = 4 + 1 + 1)
constexpr uint32_t kChunkBits = 1024; // subsequence length of the parallel Huffman decode
constexpr int kHuffThreads = 256;
constexpr uint32_t kDead = 0xFFFFFFFFu;

// Per-tile descriptor built by the host marker parse (jpeg.cu).  Offsets are relative to the batch it belongs to.
struct Tile {
  int64_t seg_off;        // entropy-coded segment = bytes [seg_off, seg_off + seg_len) of the batch's byte buffer
  int64_t coef_base;      // first 8x8 block of the tile in the batch's coefficient buffer
  int32_t seg_len;
  int32_t int_base;       // first of the tile's n_int + 1 slots in the per-interval arrays
  int32_t n_int;          // restart intervals
  int32_t ri;             // MCUs per restart interval
  int32_t chunk_base;     // first of the tile's chunk_cap slots in the per-subsequence array
  int32_t chunk_cap;
  int16_t mcux, mcuy;
  uint8_t hmax, vmax, bpm, pad0;
  uint8_t comp_h[3], comp_v[3];
  uint8_t blk_comp[kMaxBpm], blk_dy[kMaxBpm], blk_dx[kMaxBpm];
  uint8_t pad1[6];
  uint16_t qt[3][64];     // quantisation table of each component, natural order
  uint8_t hbits[6][16];   // Huffman BITS / HUFFVAL of component c: DC table at 2c, AC table at 2c + 1
  uint8_t hvals[6][256];
};

// One subsequence of a tile's entropy-coded data (kChunkBits bits of one restart interval).
struct Chunk {
  uint32_t start_pos, start_bz;   // decoder state the subsequence is decoded from: bit position, block-in-MCU << 8 | zig-zag
  uint32_t end_pos, end_bz;       // state at the first symbol boundary at or past the subsequence end (end_pos kDead: none)
  uint32_t count;                 // 8x8 blocks completed
  uint32_t err;                   // blocks completed before an invalid code (kDead: none)
  uint32_t prefix;                // blocks completed by the tile's earlier subsequences
  uint32_t interval;              // restart interval the subsequence lies in
  uint32_t next_pos, next_bz;     // synchronisation round: start state taken from the predecessor
  uint32_t dirty, pad;
};

__constant__ uint8_t kNatural[64] = {
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ------------------------------------------------------------------------------------------------------------------
// (a) byte unstuffing.  Whether a byte survives depends only on it and its neighbours, so every thread classifies its
// bytes independently and a block scan places them.  FF00 -> FF; FF D0..D7 -> restart boundary; FF FF -> fill byte;
// any other marker inside the segment is an error.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kUnstuffThreads = 256, kUnstuffPerThread = 4;

__global__ void __launch_bounds__(kUnstuffThreads) jpeg_unstuff_kernel(const Tile* __restrict__ tiles,
                                                                        const uint8_t* __restrict__ data,
                                                                        uint8_t* __restrict__ ub,
                                                                        int32_t* __restrict__ int_start,
                                                                        int32_t* __restrict__ status) {
  using Scan = cub::BlockScan<uint32_t, kUnstuffThreads>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ uint32_t s_kept, s_rst;
  __shared__ int s_err;
  const Tile& t = tiles[blockIdx.x];
  const int64_t len = t.seg_len;
  const uint8_t* src = data + t.seg_off;
  uint8_t* dst = ub + t.seg_off;
  int32_t* starts = int_start + t.int_base;
  const int n_int = t.n_int;
  if (threadIdx.x == 0) { s_kept = 0; s_rst = 0; s_err = 0; }
  __syncthreads();
  for (int64_t base = 0; base < len; base += kUnstuffThreads * kUnstuffPerThread) {
    const int64_t i0 = base + (int64_t)threadIdx.x * kUnstuffPerThread;
    uint32_t keep_mask = 0, rst_mask = 0;
    int err = 0;
    uint8_t v[kUnstuffPerThread];
#pragma unroll
    for (int j = 0; j < kUnstuffPerThread; ++j) {
      const int64_t i = i0 + j;
      v[j] = 0;
      if (i >= len) continue;
      const uint8_t x = src[i];
      v[j] = x;
      if (x == 0xFF) {
        const int nx = i + 1 < len ? src[i + 1] : -1;
        if (nx == 0x00) keep_mask |= 1u << j;
        else if (nx >= 0xD0 && nx <= 0xD7) rst_mask |= 1u << j;
        else if (nx != 0xFF) err = 1;   // another marker, or the segment ends on a bare FF
      } else if (i == 0 || src[i - 1] != 0xFF) {
        keep_mask |= 1u << j;
      }
    }
    const uint32_t mine = (uint32_t)__popc(keep_mask) | ((uint32_t)__popc(rst_mask) << 16);
    uint32_t excl, total;
    Scan(tmp).ExclusiveSum(mine, excl, total);
    if (err) s_err = 1;
    uint32_t kept = s_kept + (excl & 0xFFFF), rst = s_rst + (excl >> 16);
#pragma unroll
    for (int j = 0; j < kUnstuffPerThread; ++j) {
      if (keep_mask >> j & 1) dst[kept++] = v[j];
      if (rst_mask >> j & 1) {
        ++rst;                                             // this is restart marker number `rst` (1-based)
        const int64_t i = i0 + j;
        if ((int)rst >= n_int || src[i + 1] != 0xD0 + ((rst - 1) & 7)) s_err = 1;
        else starts[rst] = (int32_t)kept;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) { s_kept += total & 0xFFFF; s_rst += total >> 16; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    starts[0] = 0;
    starts[n_int] = (int32_t)s_kept;
    if (s_err || (int)s_rst != n_int - 1) status[blockIdx.x] = BQ_JPEG_BAD_ENTROPY_MARKER;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// (b) Huffman decode
// ------------------------------------------------------------------------------------------------------------------
struct HuffTab {
  uint16_t lut[512];      // 9-bit first level: length << 8 | symbol, 0 = code longer than 9 bits
  int32_t maxcode[18];    // jdhuff.c: largest code of each length (-1: none), maxcode[17] sentinel
  int32_t valoff[17];     // symbol index of a code of length l = code + valoff[l]
  uint8_t vals[256];
};

__device__ __forceinline__ void build_table(HuffTab& h, const uint8_t* bits, const uint8_t* vals, int lane, int nl) {
  if (lane == 0) {
    int code = 0, k = 0;
    for (int l = 1; l <= 16; ++l) {
      const int c = bits[l - 1];
      h.valoff[l] = k - code;
      h.maxcode[l] = c ? code + c - 1 : -1;
      k += c;
      code = (code + c) << 1;
    }
    h.maxcode[17] = 0x7FFFFFFF;
  }
  for (int i = lane; i < 256; i += nl) h.vals[i] = vals[i];
  __syncwarp();
  for (int i = lane; i < 512; i += nl) {
    uint16_t e = 0;
    for (int l = 1; l <= 9; ++l) {
      const int code = i >> (9 - l);
      if (code <= h.maxcode[l]) { e = (uint16_t)(l << 8 | h.vals[code + h.valoff[l]]); break; }
    }
    h.lut[i] = e;
  }
}

__device__ __forceinline__ int extend(uint32_t x, uint32_t s) {
  return (s && x < (1u << (s - 1))) ? (int)x - (1 << s) + 1 : (int)x;
}

struct RunOut { uint32_t pos, bz, count, err; };

// Decode from state (pos, bz) until the first symbol boundary at or past `stop`.  Reads only bytes below
// end_bits / 8 of this restart interval.  kWrite stores coefficients of blocks prefix + i < expected at
// coef[(prefix + i) * 64] (DC as the difference to the predictor).
template <bool kWrite>
__device__ RunOut huff_run(const HuffTab* __restrict__ tabs, const uint8_t* __restrict__ bytes, uint32_t end_bits,
                           uint32_t pos, uint32_t bz, uint32_t stop, const uint8_t* blk_comp, uint32_t bpm,
                           int16_t* __restrict__ coef, uint32_t prefix, uint32_t expected) {
  const uint32_t end_byte = end_bits >> 3;
  uint32_t bytepos = pos >> 3;
  uint64_t buf = 0;
  int nb = 0;
  auto refill = [&]() {
    while (nb <= 56) {
      const uint64_t b = bytepos < end_byte ? bytes[bytepos] : 0;
      buf |= b << (56 - nb);
      nb += 8;
      ++bytepos;
    }
  };
  refill();
  buf <<= (pos & 7);
  nb -= (int)(pos & 7);
  uint32_t blk = bz >> 8, z = bz & 0xFF, count = 0;
  RunOut o;
  o.err = kDead;
  while (pos < stop) {
    refill();
    const HuffTab& T = tabs[2 * blk_comp[blk] + (z ? 1 : 0)];
    uint32_t len, sym;
    const uint32_t e = T.lut[buf >> 55];
    if (e) {
      len = e >> 8;
      sym = e & 0xFF;
    } else {
      len = 10;
      int32_t code = (int32_t)(buf >> 54);
      while (code > T.maxcode[len]) { ++len; code = (int32_t)(buf >> (64 - len)); }
      if (len > 16) {
        if (end_bits - pos >= 16) o.err = count;      // a code that exists in no table: invalid data
        o.pos = kDead;
        o.bz = 0;
        o.count = count;
        return o;
      }
      sym = T.vals[(code + T.valoff[len]) & 0xFF];
    }
    const uint32_t s = z ? (sym & 15) : sym;
    if (pos + len + s > end_bits) break;                 // runs past the end of the interval
    buf <<= len;
    pos += len;
    nb -= (int)len;
    int v = 0;
    if (s) {
      v = extend((uint32_t)(buf >> (64 - s)), s);
      buf <<= s;
      pos += s;
      nb -= (int)s;
    }
    const uint32_t bi = prefix + count;
    if (z == 0) {
      if (kWrite && bi < expected) coef[(size_t)bi * 64] = (int16_t)v;
      z = 1;
    } else if (s == 0) {
      z = (sym >> 4) == 15 ? z + 16 : 64;              // ZRL / EOB
    } else {
      z += sym >> 4;
      // jdhuff.c writes a run past the block end at natural position 63 (jpeg_natural_order's guard entries)
      if (kWrite && bi < expected) coef[(size_t)bi * 64 + (z < 64 ? kNatural[z] : 63)] = (int16_t)v;
      ++z;
    }
    if (z >= 64) {
      z = 0;
      ++count;
      blk = blk + 1 == bpm ? 0 : blk + 1;
    }
  }
  if (pos < stop) { o.pos = kDead; o.bz = 0; }         // ran out of bits
  else { o.pos = pos; o.bz = blk << 8 | z; }
  o.count = count;
  return o;
}

__device__ __forceinline__ uint32_t find_interval(const int32_t* ichunk, int n_int, uint32_t c) {
  int lo = 0, hi = n_int - 1;                           // last k with ichunk[k] <= c
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((uint32_t)ichunk[mid] <= c) lo = mid; else hi = mid - 1;
  }
  return (uint32_t)lo;
}

// stats[tile * 3 + {0, 1, 2}] = subsequences, synchronisation rounds, subsequences decoded again
__global__ void __launch_bounds__(kHuffThreads) jpeg_huffman_kernel(const Tile* __restrict__ tiles,
                                                                     const uint8_t* __restrict__ ub,
                                                                     const int32_t* __restrict__ int_start,
                                                                     int32_t* __restrict__ int_chunk,
                                                                     Chunk* __restrict__ chunks,
                                                                     int16_t* __restrict__ coef,
                                                                     int32_t* __restrict__ status,
                                                                     int32_t* __restrict__ stats) {
  using Scan = cub::BlockScan<uint32_t, kHuffThreads>;
  __shared__ HuffTab tabs[6];
  __shared__ typename Scan::TempStorage tmp;
  __shared__ uint32_t s_carry, s_redecoded;
  __shared__ uint8_t s_blk_comp[kMaxBpm];
  const Tile& t = tiles[blockIdx.x];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (status[blockIdx.x] != 0) return;                  // the unstuffing pass already rejected the tile
  if (warp < 6) build_table(tabs[warp], t.hbits[warp], t.hvals[warp], lane, 32);
  if (threadIdx.x < kMaxBpm) s_blk_comp[threadIdx.x] = t.blk_comp[threadIdx.x];
  const int n_int = t.n_int;
  const uint32_t bpm = t.bpm, ri = (uint32_t)t.ri, mcus = (uint32_t)t.mcux * (uint32_t)t.mcuy;
  const int32_t* starts = int_start + t.int_base;
  int32_t* ichunk = int_chunk + t.int_base;
  Chunk* ch = chunks + t.chunk_base;
  const uint8_t* bytes = ub + t.seg_off;
  int16_t* tcoef = coef + (size_t)t.coef_base * 64;

  // subsequences per restart interval -> first subsequence of each interval
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int k0 = 0; k0 < n_int; k0 += kHuffThreads) {
    const int k = k0 + threadIdx.x;
    uint32_t nch = 0;
    if (k < n_int) {
      const uint32_t bits = (uint32_t)(starts[k + 1] - starts[k]) * 8u;
      nch = bits ? (bits + kChunkBits - 1) / kChunkBits : 1;
    }
    uint32_t excl, total;
    Scan(tmp).ExclusiveSum(nch, excl, total);
    if (k < n_int) ichunk[k] = (int32_t)(s_carry + excl);
    __syncthreads();
    if (threadIdx.x == 0) s_carry += total;
    __syncthreads();
  }
  const uint32_t nchunks = s_carry;
  if (threadIdx.x == 0) ichunk[n_int] = (int32_t)nchunks;
  if (nchunks > (uint32_t)t.chunk_cap) {                // cannot happen for a segment the unstuffing pass accepted
    if (threadIdx.x == 0) status[blockIdx.x] = BQ_JPEG_BAD_ENTROPY_MARKER;
    return;
  }
  __syncthreads();

  // first pass: interval starts are known-good, every other subsequence starts speculatively at a block start
  for (uint32_t c = threadIdx.x; c < nchunks; c += kHuffThreads) {
    const uint32_t k = find_interval(ichunk, n_int, c);
    const uint32_t j = c - (uint32_t)ichunk[k];
    const uint32_t b0 = (uint32_t)starts[k] * 8u, b1 = (uint32_t)starts[k + 1] * 8u;
    const uint32_t sp = b0 + j * kChunkBits;
    const uint32_t stop = min(sp + kChunkBits, b1);
    const RunOut o = huff_run<false>(tabs, bytes, b1, sp, 0, stop, s_blk_comp, bpm, nullptr, 0, 0);
    Chunk q;
    q.start_pos = sp; q.start_bz = 0; q.end_pos = o.pos; q.end_bz = o.bz; q.count = o.count; q.err = o.err;
    q.prefix = 0; q.interval = k; q.next_pos = 0; q.next_bz = 0; q.dirty = 0; q.pad = 0;
    ch[c] = q;
  }
  __syncthreads();

  // synchronisation: a subsequence whose predecessor ended in a different state than it started from is decoded
  // again from that state, until no start changes.  The first subsequence of every interval is exact, so round r
  // fixes at least subsequence r of each interval: one that never falls into step is still decoded correctly.
  uint32_t rounds = 0, redecoded = 0;
  while (true) {
    bool any = false;
    for (uint32_t c = threadIdx.x; c < nchunks; c += kHuffThreads) {   // read every predecessor before any redecode
      Chunk& q = ch[c];
      if ((uint32_t)ichunk[q.interval] == c) continue;
      const uint32_t ep = ch[c - 1].end_pos, eb = ch[c - 1].end_bz;
      if (ep != kDead && (ep != q.start_pos || eb != q.start_bz)) {
        q.next_pos = ep;
        q.next_bz = eb;
        q.dirty = 1;
        any = true;
      }
    }
    if (!__syncthreads_or(any)) break;
    ++rounds;
    for (uint32_t c = threadIdx.x; c < nchunks; c += kHuffThreads) {
      Chunk& q = ch[c];
      if (!q.dirty) continue;
      const uint32_t k = q.interval;
      const uint32_t j = c - (uint32_t)ichunk[k];
      const uint32_t b1 = (uint32_t)starts[k + 1] * 8u;
      const uint32_t stop = min((uint32_t)starts[k] * 8u + (j + 1) * kChunkBits, b1);
      const RunOut o = huff_run<false>(tabs, bytes, b1, q.next_pos, q.next_bz, stop, s_blk_comp, bpm, nullptr, 0, 0);
      q.start_pos = q.next_pos; q.start_bz = q.next_bz; q.dirty = 0;
      q.end_pos = o.pos; q.end_bz = o.bz; q.count = o.count; q.err = o.err;
      ++redecoded;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) s_redecoded = 0;
  __syncthreads();
  atomicAdd(&s_redecoded, redecoded);

  // blocks completed before each subsequence (tile-wide exclusive scan; per interval by difference)
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t c0 = 0; c0 < nchunks; c0 += kHuffThreads) {
    const uint32_t c = c0 + threadIdx.x;
    const uint32_t cnt = c < nchunks ? ch[c].count : 0;
    uint32_t excl, total;
    Scan(tmp).ExclusiveSum(cnt, excl, total);
    if (c < nchunks) ch[c].prefix = s_carry + excl;
    __syncthreads();
    if (threadIdx.x == 0) s_carry += total;
    __syncthreads();
  }
  const uint32_t all_blocks = s_carry;
  // per interval: enough blocks, and no invalid code before the last expected block
  int bad = 0;
  for (int k = threadIdx.x; k < n_int; k += kHuffThreads) {
    const uint32_t first = (uint32_t)ichunk[k], next = (uint32_t)ichunk[k + 1];
    const uint32_t p1 = next < nchunks ? ch[next].prefix : all_blocks;
    const uint32_t expected = min(ri, mcus - (uint32_t)k * ri) * bpm;
    if (p1 - ch[first].prefix < expected) bad = max(bad, (int)BQ_JPEG_TRUNCATED_DATA);
  }
  for (uint32_t c = threadIdx.x; c < nchunks; c += kHuffThreads) {
    const Chunk q = ch[c];
    if (q.err == kDead) continue;
    const uint32_t k = q.interval;
    const uint32_t expected = min(ri, mcus - k * ri) * bpm;
    if (q.prefix - ch[ichunk[k]].prefix + q.err < expected) bad = BQ_JPEG_INVALID_CODE;
  }
  const int invalid = __syncthreads_or(bad == BQ_JPEG_INVALID_CODE);
  const int truncated = __syncthreads_or(bad != 0);
  if (threadIdx.x == 0) {
    stats[blockIdx.x * 3 + 0] = (int32_t)nchunks;
    stats[blockIdx.x * 3 + 1] = (int32_t)rounds;
    stats[blockIdx.x * 3 + 2] = (int32_t)s_redecoded;
  }
  if (invalid || truncated) {
    if (threadIdx.x == 0) status[blockIdx.x] = invalid ? BQ_JPEG_INVALID_CODE : BQ_JPEG_TRUNCATED_DATA;
    return;
  }

  // writing pass: every subsequence decodes again from its exact start and stores its blocks' coefficients
  for (uint32_t c = threadIdx.x; c < nchunks; c += kHuffThreads) {
    const Chunk q = ch[c];
    const uint32_t k = q.interval;
    const uint32_t j = c - (uint32_t)ichunk[k];
    const uint32_t b1 = (uint32_t)starts[k + 1] * 8u;
    const uint32_t stop = min((uint32_t)starts[k] * 8u + (j + 1) * kChunkBits, b1);
    const uint32_t expected = min(ri, mcus - k * ri) * bpm;
    huff_run<true>(tabs, bytes, b1, q.start_pos, q.start_bz, stop, s_blk_comp, bpm,
                   tcoef + (size_t)k * ri * bpm * 64, q.prefix - ch[ichunk[k]].prefix, expected);
  }
  __syncthreads();

  // DC prediction: running sum of the differences per component, restarted at every interval (warp c: component c)
  if (warp < 3) {
    const int cc = warp;
    int off = 0, nk = 0;
    for (uint32_t b = 0; b < bpm; ++b) {
      if (t.blk_comp[b] < cc) ++off;
      if (t.blk_comp[b] == cc) ++nk;
    }
    for (int k = 0; k < n_int; ++k) {
      const uint32_t m0 = (uint32_t)k * ri, nm = min(ri, mcus - m0);
      const uint32_t nblk = nm * nk;
      int carry = 0;
      for (uint32_t i0 = 0; i0 < nblk; i0 += 32) {
        const uint32_t i = i0 + lane;
        size_t idx = 0;
        int v = 0;
        if (i < nblk) {
          idx = ((size_t)(m0 + i / nk) * bpm + off + i % nk) * 64;
          v = tcoef[idx];
        }
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int u = __shfl_up_sync(0xFFFFFFFFu, v, d);
          if (lane >= d) v += u;
        }
        v += carry;
        if (i < nblk) tcoef[idx] = (int16_t)v;           // jdhuff.c keeps the predictor as int, stores a JCOEF
        carry = __shfl_sync(0xFFFFFFFFu, v, 31);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// (c) dequantisation + jidctint.c jpeg_idct_islow or jidctfst.c jpeg_idct_ifast.  Eight threads per block: thread r
// transforms column r, then row r.  All arithmetic is exact integer; the range limit is the saturating one of
// libjpeg-turbo's SIMD IDCT, equal to the C table lookup wherever |value| < 512.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kIdctThreads = 256, kIdctBlocks = kIdctThreads / 8;

enum class Idct { kIslow, kIfast };

// jddctmgr.c aanscales (natural order): 16384 * s(row) * s(col), s(0) = 1, s(k) = sqrt(2) cos(k pi / 16)
__constant__ int32_t kAanScales[64] = {
    16384, 22725, 21407, 19266, 16384, 12873, 8867,  4520,  22725, 31521, 29692, 26722, 22725, 17855, 12299, 6270,
    21407, 29692, 27969, 25172, 21407, 16819, 11585, 5906,  19266, 26722, 25172, 22654, 19266, 15137, 10426, 5315,
    16384, 22725, 21407, 19266, 16384, 12873, 8867,  4520,  12873, 17855, 16819, 15137, 12873, 10114, 6967,  3552,
    8867,  12299, 11585, 10426, 8867,  6967,  4799,  2446,  4520,  6270,  5906,  5315,  4520,  3552,  2446,  1247};

__device__ __forceinline__ void islow_1d(int32_t i0, int32_t i1, int32_t i2, int32_t i3, int32_t i4, int32_t i5,
                                         int32_t i6, int32_t i7, int shift, int32_t* o) {
  int32_t z2 = i2, z3 = i6;
  int32_t z1 = (z2 + z3) * 4433;
  int32_t tmp2 = z1 + z3 * -15137;
  int32_t tmp3 = z1 + z2 * 6270;
  int32_t tmp0 = (i0 + i4) * 8192;
  int32_t tmp1 = (i0 - i4) * 8192;
  const int32_t t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
  tmp0 = i7; tmp1 = i5; tmp2 = i3; tmp3 = i1;
  z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2;
  int32_t z4 = tmp1 + tmp3;
  const int32_t z5 = (z3 + z4) * 9633;
  tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
  z1 *= -7373; z2 *= -20995; z3 = z3 * -16069 + z5; z4 = z4 * -3196 + z5;
  tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
  const int32_t r = 1 << (shift - 1);
  o[0] = (t10 + tmp3 + r) >> shift;
  o[7] = (t10 - tmp3 + r) >> shift;
  o[1] = (t11 + tmp2 + r) >> shift;
  o[6] = (t11 - tmp2 + r) >> shift;
  o[2] = (t12 + tmp1 + r) >> shift;
  o[5] = (t12 - tmp1 + r) >> shift;
  o[3] = (t13 + tmp0 + r) >> shift;
  o[4] = (t13 - tmp0 + r) >> shift;
}

// jidctfst.c: CONST_BITS 8 multiplies that truncate (no USE_ACCURATE_ROUNDING); the product is taken in 64 bits as
// libjpeg-turbo's JLONG is
__device__ __forceinline__ int32_t ifast_mul(int32_t v, int32_t c) { return (int32_t)(((int64_t)v * c) >> 8); }

// One jpeg_idct_ifast pass.  It keeps the scale of its input: the caller shifts the row pass right by PASS1_BITS + 3.
__device__ __forceinline__ void ifast_1d(int32_t i0, int32_t i1, int32_t i2, int32_t i3, int32_t i4, int32_t i5,
                                         int32_t i6, int32_t i7, int32_t* o) {
  const int32_t t10 = i0 + i4, t11 = i0 - i4, t13 = i2 + i6;
  const int32_t t12 = ifast_mul(i2 - i6, 362) - t13;
  const int32_t e0 = t10 + t13, e3 = t10 - t13, e1 = t11 + t12, e2 = t11 - t12;
  const int32_t z13 = i5 + i3, z10 = i5 - i3, z11 = i1 + i7, z12 = i1 - i7;
  const int32_t o7 = z11 + z13;
  const int32_t o11 = ifast_mul(z11 - z13, 362);
  const int32_t z5 = ifast_mul(z10 + z12, 473);
  const int32_t o10 = ifast_mul(z12, 277) - z5;
  const int32_t o12 = ifast_mul(z10, -669) + z5;
  const int32_t o6 = o12 - o7, o5 = o11 - o6, o4 = o10 + o5;
  o[0] = e0 + o7;
  o[7] = e0 - o7;
  o[1] = e1 + o6;
  o[6] = e1 - o6;
  o[2] = e2 + o5;
  o[5] = e2 - o5;
  o[3] = e3 - o4;
  o[4] = e3 + o4;
}

// jddctmgr.c: the IFAST multiplier of quantisation table entry i (natural order), DESCALE by 12 bits and the
// IFAST_MULT_TYPE (short) cast.  q * aan < 2^31 for every 16-bit q.
__device__ __forceinline__ int32_t ifast_multiplier(uint32_t q, int i) {
  return (int16_t)((q * (uint32_t)kAanScales[i] + 2048u) >> 12);
}

template <Idct kMethod>
__global__ void __launch_bounds__(kIdctThreads) jpeg_idct_kernel(const Tile* __restrict__ tiles,
                                                                  const int16_t* __restrict__ coef,
                                                                  const int32_t* __restrict__ status,
                                                                  uint8_t* __restrict__ planes, int pitch) {
  __shared__ int32_t ws[kIdctBlocks][8][9];
  const int tile = blockIdx.y;
  if (status[tile] != 0) return;
  const Tile& t = tiles[tile];
  const int g = threadIdx.x >> 3, r = threadIdx.x & 7;
  const int nblocks = (int)t.mcux * t.mcuy * t.bpm;
  const int b = blockIdx.x * kIdctBlocks + g;
  if (b >= nblocks) return;                              // whole 8-thread groups leave together
  const unsigned gmask = 0xFFu << (threadIdx.x & 24);
  const int mcu = b / t.bpm, j = b - mcu * t.bpm;
  const int comp = t.blk_comp[j];
  const int by = (mcu / t.mcux) * t.comp_v[comp] + t.blk_dy[j];
  const int bx = (mcu % t.mcux) * t.comp_h[comp] + t.blk_dx[j];
  const int16_t* cb = coef + ((size_t)t.coef_base + b) * 64;
  const uint16_t* q = t.qt[comp];
  int32_t in[8], out[8];
  if constexpr (kMethod == Idct::kIslow) {
#pragma unroll
    for (int k = 0; k < 8; ++k) in[k] = (int32_t)cb[k * 8 + r] * (int32_t)q[k * 8 + r];
    islow_1d(in[0], in[1], in[2], in[3], in[4], in[5], in[6], in[7], 11, out);
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k) in[k] = (int32_t)cb[k * 8 + r] * ifast_multiplier(q[k * 8 + r], k * 8 + r);
    ifast_1d(in[0], in[1], in[2], in[3], in[4], in[5], in[6], in[7], out);
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) ws[g][k][r] = out[k];
  __syncwarp(gmask);
  if constexpr (kMethod == Idct::kIslow) {
    islow_1d(ws[g][r][0], ws[g][r][1], ws[g][r][2], ws[g][r][3], ws[g][r][4], ws[g][r][5], ws[g][r][6], ws[g][r][7],
             18, out);
  } else {
    ifast_1d(ws[g][r][0], ws[g][r][1], ws[g][r][2], ws[g][r][3], ws[g][r][4], ws[g][r][5], ws[g][r][6], ws[g][r][7],
             out);
#pragma unroll
    for (int k = 0; k < 8; ++k) out[k] >>= 5;           // PASS1_BITS + 3, truncating
  }
  uint32_t lo = 0, hi = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    lo |= (uint32_t)min(max(out[k] + 128, 0), 255) << (8 * k);
    hi |= (uint32_t)min(max(out[k + 4] + 128, 0), 255) << (8 * k);
  }
  uint8_t* dst = planes + ((size_t)tile * 3 + comp) * pitch * pitch + (size_t)(by * 8 + r) * pitch + bx * 8;
  *reinterpret_cast<uint2*>(dst) = make_uint2(lo, hi);
}

// ------------------------------------------------------------------------------------------------------------------
// (d) jdsample.c fancy upsampling (h2v1 / h2v2, edge samples replicated, odd widths cut at the downsampled width) or,
// without fancy upsampling, jdmerge.c's replicated chroma (each chroma sample covers its 2x1 / 2x2 output pixels), and
// jdcolor.c ycc_rgb_convert (jdmerge.c uses the same tables), one thread per output pixel.
// ------------------------------------------------------------------------------------------------------------------
enum class Upsample { kFancy, kReplicate };

template <Upsample kUp>
__device__ __forceinline__ int chroma(const uint8_t* p, int pitch, int mode, int y, int x, int dw, int dh) {
  if (mode == 0) return p[y * pitch + x];
  if constexpr (kUp == Upsample::kReplicate) return p[(mode == 1 ? y : y >> 1) * pitch + (x >> 1)];
  const int i = x >> 1, odd = x & 1;
  const int ni = odd ? min(i + 1, dw - 1) : max(i - 1, 0);
  if (mode == 1) {
    const uint8_t* row = p + y * pitch;
    return (3 * row[i] + row[ni] + 1 + odd) >> 2;
  }
  const int rr = y >> 1;
  const int far = (y & 1) ? min(rr + 1, dh - 1) : max(rr - 1, 0);
  const uint8_t* near_row = p + rr * pitch;
  const uint8_t* far_row = p + far * pitch;
  const int cs = 3 * near_row[i] + far_row[i];
  const int cn = 3 * near_row[ni] + far_row[ni];
  return (3 * cs + cn + 8 - odd) >> 4;
}

template <Upsample kUp>
__global__ void __launch_bounds__(256) jpeg_color_kernel(const Tile* __restrict__ tiles, const uint8_t* __restrict__ planes,
                                                         const int32_t* __restrict__ status, int pitch, int px,
                                                         uint8_t* __restrict__ out) {
  const int tile = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= px * px) return;
  uint8_t* o = out + ((size_t)tile * px * px + idx) * 3;
  if (status[tile] != 0) { o[0] = o[1] = o[2] = 0; return; }
  const Tile& t = tiles[tile];
  const int y = idx / px, x = idx - y * px;
  const int mode = t.hmax == 1 ? 0 : (t.vmax == 1 ? 1 : 2);
  const int dw = (px + t.hmax - 1) / t.hmax, dh = (px + t.vmax - 1) / t.vmax;
  const uint8_t* p0 = planes + (size_t)tile * 3 * pitch * pitch;
  const int Y = p0[y * pitch + x];
  const int cb = chroma<kUp>(p0 + (size_t)pitch * pitch, pitch, mode, y, x, dw, dh) - 128;
  const int cr = chroma<kUp>(p0 + (size_t)2 * pitch * pitch, pitch, mode, y, x, dw, dh) - 128;
  const int R = Y + ((91881 * cr + 32768) >> 16);
  const int G = Y + ((-46802 * cr - 22554 * cb + 32768) >> 16);
  const int B = Y + ((116130 * cb + 32768) >> 16);
  o[0] = (uint8_t)min(max(R, 0), 255);
  o[1] = (uint8_t)min(max(G, 0), 255);
  o[2] = (uint8_t)min(max(B, 0), 255);
}

}  // namespace jpeg
}  // namespace bq
