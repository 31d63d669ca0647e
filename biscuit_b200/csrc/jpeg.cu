// Baseline-JPEG tiles on the GPU: the host marker parse into per-tile descriptors, the layout of their decode scratch
// and the four decode launches of jpeg_sm100.cuh, driven by encoded.cu, and the bq_jpeg_* entry points.
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "../../include/biscuit_b200.h"
#include "encoded.cuh"
#include "jpeg_sm100.cuh"

using bq::jpeg::Tile;

namespace {

const uint8_t kNaturalHost[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                  35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                  58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// Marker parse of one file b[0, len) of which the first `avail` bytes are at hand (tail2 = its last two bytes).
// Returns BQ_JPEG_* (t filled on BQ_JPEG_OK; t.seg_off relative to the file start) or bq_encoded::kNeedMore.
int parse_tile(const uint8_t* b, int64_t len, int64_t avail, const uint8_t* tail2, int px, Tile& t) {
  memset(&t, 0, sizeof(t));
#define NEED(k)                                        \
  do {                                                 \
    if ((int64_t)(k) > len) return BQ_JPEG_TRUNCATED_HEADER; \
    if ((int64_t)(k) > avail) return bq_encoded::kNeedMore; \
  } while (0)
  NEED(2);
  if (b[0] != 0xFF || b[1] != 0xD8) return BQ_JPEG_NOT_JPEG;
  bool qdef[4] = {}, hdef[2][4] = {}, sof = false, jfif = false;
  uint16_t q[4][64];
  uint8_t hb[2][4][16], hv[2][4][256];
  int adobe_transform = -1, ri = 0;
  int ids[3] = {}, hs[3] = {}, vs[3] = {}, tq[3] = {};
  int64_t i = 2;
  for (;;) {
    NEED(i + 2);
    if (b[i] != 0xFF) return BQ_JPEG_BAD_HEADER;
    while (b[i + 1] == 0xFF) { ++i; NEED(i + 2); }     // fill bytes
    const int m = b[i + 1];
    i += 2;
    if (m == 0xD9 || m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01 || m == 0x00) return BQ_JPEG_BAD_HEADER;
    NEED(i + 2);
    const int L = b[i] << 8 | b[i + 1];
    if (L < 2) return BQ_JPEG_BAD_HEADER;
    NEED(i + L);
    const uint8_t* s = b + i + 2;
    const int sl = L - 2;
    if (m == 0xC9 || m == 0xCA || m == 0xCB || m == 0xCC || m == 0xCD || m == 0xCE || m == 0xCF) return BQ_JPEG_ARITHMETIC;
    if (m == 0xC2 || m == 0xC6) return BQ_JPEG_PROGRESSIVE;
    if (m == 0xC3 || m == 0xC5 || m == 0xC7 || m == 0xDE) return BQ_JPEG_LOSSLESS;
    if (m == 0xC0 || m == 0xC1) {
      if (sof || sl < 6) return BQ_JPEG_BAD_HEADER;
      if (s[0] != 8) return BQ_JPEG_PRECISION;
      const int nf = s[5];
      if (sl < 6 + 3 * nf) return BQ_JPEG_BAD_HEADER;
      if (nf == 1) return BQ_JPEG_GRAYSCALE;
      if (nf == 4) return BQ_JPEG_CMYK;
      if (nf != 3) return BQ_JPEG_COMPONENTS;
      if ((s[1] << 8 | s[2]) != px || (s[3] << 8 | s[4]) != px) return BQ_JPEG_SIZE;
      for (int c = 0; c < 3; ++c) {
        ids[c] = s[6 + 3 * c];
        hs[c] = s[7 + 3 * c] >> 4;
        vs[c] = s[7 + 3 * c] & 15;
        tq[c] = s[8 + 3 * c];
        if (tq[c] > 3) return BQ_JPEG_BAD_HEADER;
      }
      sof = true;
    } else if (m == 0xC4) {
      int k = 0;
      while (k < sl) {
        if (k + 17 > sl) return BQ_JPEG_BAD_TABLE;
        const int tc = s[k] >> 4, th = s[k] & 15;
        if (tc > 1 || th > 3) return BQ_JPEG_BAD_TABLE;
        int count = 0, code = 0;
        for (int l = 1; l <= 16; ++l) {
          count += s[k + l];
          code += s[k + l];
          if (code > (1 << l)) return BQ_JPEG_BAD_TABLE;   // jdhuff.c: codes must fit their length
          code <<= 1;
        }
        if (count > 256 || k + 17 + count > sl) return BQ_JPEG_BAD_TABLE;
        memcpy(hb[tc][th], s + k + 1, 16);
        memset(hv[tc][th], 0, 256);
        memcpy(hv[tc][th], s + k + 17, count);
        if (tc == 0)
          for (int j = 0; j < count; ++j)
            if (hv[tc][th][j] > 15) return BQ_JPEG_BAD_TABLE;
        hdef[tc][th] = true;
        k += 17 + count;
      }
    } else if (m == 0xDB) {
      int k = 0;
      while (k < sl) {
        const int pq = s[k] >> 4, tqi = s[k] & 15;
        if (pq > 1 || tqi > 3) return BQ_JPEG_BAD_TABLE;
        const int n = pq ? 128 : 64;
        if (k + 1 + n > sl) return BQ_JPEG_BAD_TABLE;
        for (int z = 0; z < 64; ++z)
          q[tqi][kNaturalHost[z]] = pq ? (uint16_t)(s[k + 1 + 2 * z] << 8 | s[k + 2 + 2 * z]) : s[k + 1 + z];
        qdef[tqi] = true;
        k += 1 + n;
      }
    } else if (m == 0xDD) {
      if (sl != 2) return BQ_JPEG_BAD_HEADER;
      ri = s[0] << 8 | s[1];
    } else if (m == 0xE0) {
      if (sl >= 5 && memcmp(s, "JFIF\0", 5) == 0) jfif = true;
    } else if (m == 0xEE) {
      if (sl >= 12 && memcmp(s, "Adobe", 5) == 0) adobe_transform = s[11];
    } else if (m == 0xDA) {
      if (!sof || sl < 1) return BQ_JPEG_BAD_HEADER;
      const int ns = s[0];
      if (ns != 3 || sl != 1 + 2 * ns + 3) return BQ_JPEG_BAD_HEADER;   // one interleaved scan of all components
      int td[3], ta[3];
      for (int c = 0; c < 3; ++c) {
        if (s[1 + 2 * c] != ids[c]) return BQ_JPEG_BAD_HEADER;
        td[c] = s[2 + 2 * c] >> 4;
        ta[c] = s[2 + 2 * c] & 15;
        if (td[c] > 3 || ta[c] > 3) return BQ_JPEG_BAD_HEADER;
      }
      if (s[7] != 0 || s[8] != 63 || s[9] != 0) return BQ_JPEG_BAD_HEADER;
      for (int c = 0; c < 3; ++c) {
        if (!qdef[tq[c]]) return BQ_JPEG_MISSING_DQT;
        if (!hdef[0][td[c]] || !hdef[1][ta[c]]) return BQ_JPEG_MISSING_DHT;
      }
      if (adobe_transform == 0 || (!jfif && adobe_transform < 0 && ids[0] == 'R' && ids[1] == 'G' && ids[2] == 'B'))
        return BQ_JPEG_COLORSPACE;
      const bool chroma_1x1 = hs[1] == 1 && vs[1] == 1 && hs[2] == 1 && vs[2] == 1;
      if (!chroma_1x1 || !((hs[0] == 1 && vs[0] == 1) || (hs[0] == 2 && vs[0] == 1) || (hs[0] == 2 && vs[0] == 2)))
        return BQ_JPEG_SAMPLING;
      const int64_t start = i + L;
      if (len < start + 2 || tail2[0] != 0xFF || tail2[1] != 0xD9) return BQ_JPEG_TRUNCATED_DATA;
      const int64_t seg = len - 2 - start;
      if (seg > (1 << 28)) return BQ_JPEG_BAD_HEADER;
      t.seg_off = start;
      t.seg_len = (int32_t)seg;
      t.hmax = (uint8_t)hs[0];
      t.vmax = (uint8_t)vs[0];
      t.mcux = (int16_t)((px + 8 * hs[0] - 1) / (8 * hs[0]));
      t.mcuy = (int16_t)((px + 8 * vs[0] - 1) / (8 * vs[0]));
      int bpm = 0;
      for (int c = 0; c < 3; ++c) {
        t.comp_h[c] = (uint8_t)hs[c];
        t.comp_v[c] = (uint8_t)vs[c];
        for (int dy = 0; dy < vs[c]; ++dy)
          for (int dx = 0; dx < hs[c]; ++dx, ++bpm) {
            t.blk_comp[bpm] = (uint8_t)c;
            t.blk_dy[bpm] = (uint8_t)dy;
            t.blk_dx[bpm] = (uint8_t)dx;
          }
        memcpy(t.qt[c], q[tq[c]], sizeof(t.qt[c]));
        memcpy(t.hbits[2 * c], hb[0][td[c]], 16);
        memcpy(t.hvals[2 * c], hv[0][td[c]], 256);
        memcpy(t.hbits[2 * c + 1], hb[1][ta[c]], 16);
        memcpy(t.hvals[2 * c + 1], hv[1][ta[c]], 256);
      }
      t.bpm = (uint8_t)bpm;
      const int mcus = (int)t.mcux * t.mcuy;
      t.ri = ri ? ri : mcus;
      t.n_int = (mcus + t.ri - 1) / t.ri;
      t.chunk_cap = (int32_t)(((int64_t)seg * 8 + bq::jpeg::kChunkBits - 1) / bq::jpeg::kChunkBits) + t.n_int;
      return BQ_JPEG_OK;
    }
    i += L;
  }
#undef NEED
}

const char* status_string(int32_t s) {
  switch (s) {
    case BQ_JPEG_OK: return "ok";
    case BQ_JPEG_NOT_JPEG: return "not a JPEG file (no SOI marker)";
    case BQ_JPEG_TRUNCATED_HEADER: return "file ends inside its headers";
    case BQ_JPEG_PROGRESSIVE: return "progressive JPEG is not supported (baseline / extended sequential only)";
    case BQ_JPEG_ARITHMETIC: return "arithmetic-coded JPEG is not supported (Huffman only)";
    case BQ_JPEG_LOSSLESS: return "lossless or hierarchical JPEG is not supported";
    case BQ_JPEG_PRECISION: return "sample precision is not 8 bits";
    case BQ_JPEG_GRAYSCALE: return "grayscale JPEG (1 component) is not supported: 3 components (YCbCr) expected";
    case BQ_JPEG_CMYK: return "CMYK / YCCK JPEG (4 components) is not supported: 3 components (YCbCr) expected";
    case BQ_JPEG_COMPONENTS: return "unsupported number of components: 3 (YCbCr) expected";
    case BQ_JPEG_SIZE: return "image size differs from the model's tile size";
    case BQ_JPEG_SAMPLING: return "unsupported sampling factors (4:4:4, 4:2:2 or 4:2:0 expected)";
    case BQ_JPEG_MISSING_DQT: return "a quantisation table the frame uses is missing (no DQT)";
    case BQ_JPEG_MISSING_DHT: return "a Huffman table the scan uses is missing (no DHT)";
    case BQ_JPEG_BAD_TABLE: return "malformed DQT or DHT segment";
    case BQ_JPEG_BAD_HEADER: return "malformed or unsupported marker structure (missing SOF / SOS, unexpected marker, "
                                    "non-interleaved or non-sequential scan)";
    case BQ_JPEG_COLORSPACE: return "3 components that are not YCbCr (RGB JPEG) are not supported";
    case BQ_JPEG_BAD_ENTROPY_MARKER: return "unexpected marker or wrong RSTn sequence inside the entropy-coded data";
    case BQ_JPEG_INVALID_CODE: return "invalid Huffman code in the entropy-coded data";
    case BQ_JPEG_TRUNCATED_DATA: return "entropy-coded data truncated (ends before the last MCU or has no EOI marker)";
    default: return "unknown status";
  }
}


// Decode state of one caller: the driver's, plus the JPEG decode scratch sized for the largest group.
struct Jpeg final : bq_encoded {
  DevBuf ub, intv, ichunk, chunks, coef, planes, stats;
  int64_t max_int = 0, max_chunks = 0, max_blocks = 0, max_tile_blocks = 0;
  int64_t last_stats[4] = {};

  const char* name() const override { return "JPEG"; }
  int32_t known_flags() const override { return BQ_JPEG_IDCT_IFAST | BQ_JPEG_REPLICATE_CHROMA; }
  size_t desc_bytes() const override { return sizeof(Tile); }
  int head_bytes() const override { return 2048; }
  bool px_ok(int px) const override { return px >= 16 && px <= 4096; }
  int parse(const uint8_t* b, int64_t len, int64_t avail, const uint8_t* tail2, int px, void* desc) const override {
    return parse_tile(b, len, avail, tail2, px, *(Tile*)desc);
  }
  const char* status_string(int32_t code) const override { return ::status_string(code); }

  // every base is relative to the group
  int layout(bq_ctx* ctx) override {
    Tile* tiles = (Tile*)desc_host;
    max_int = max_chunks = max_blocks = max_tile_blocks = 0;
    for (int64_t g = 0; g < n_groups(); ++g) {
      const int64_t i0 = g * group, i1 = group_end(g);
      int64_t ni = 0, nc = 0, nbk = 0;
      for (int64_t i = i0; i < i1; ++i) {
        Tile& t = tiles[i];
        t.seg_off += offs[i] - offs[i0];
        t.int_base = (int32_t)ni;
        t.chunk_base = (int32_t)nc;
        t.coef_base = nbk;
        const int64_t blocks = (int64_t)t.mcux * t.mcuy * t.bpm;
        ni += t.n_int + 1;
        nc += t.chunk_cap;
        nbk += blocks;
        max_tile_blocks = std::max(max_tile_blocks, blocks);
      }
      if (nc > INT32_MAX || ni > INT32_MAX) return bq_fail(ctx, BQ_ERR_ARG, "bq_jpeg: group too large");
      max_int = std::max(max_int, ni);
      max_chunks = std::max(max_chunks, nc);
      max_blocks = std::max(max_blocks, nbk);
    }
    const size_t pitch = bq_align_up((size_t)px, 16);
    const int64_t gmax = std::min(n, group);
    int rc;
    if ((rc = bq_alloc(ctx, ub, max_bytes + 16)) || (rc = bq_alloc(ctx, intv, (size_t)max_int * 4)) ||
        (rc = bq_alloc(ctx, ichunk, (size_t)max_int * 4)) ||
        (rc = bq_alloc(ctx, chunks, (size_t)max_chunks * sizeof(bq::jpeg::Chunk))) ||
        (rc = bq_alloc(ctx, coef, (size_t)max_blocks * 128)) ||
        (rc = bq_alloc(ctx, planes, (size_t)gmax * 3 * pitch * pitch)) ||
        (rc = bq_alloc(ctx, stats, (size_t)std::max<int64_t>(n, 1) * 12)))
      return rc;
    return BQ_OK;
  }

  int launch(bq_ctx* ctx, int64_t i0, int nb, const uint8_t* src, const void* desc_dev, int32_t* status,
             uint8_t* out) override {
    namespace J = bq::jpeg;
    const int pitch = (int)bq_align_up((size_t)px, 16);
    const Tile* d = (const Tile*)desc_dev;
    const Tile* tiles = (const Tile*)desc_host;
    int32_t* st = (int32_t*)stats.p + 3 * i0;
    int64_t blocks = 0;
    for (int64_t i = i0; i < i0 + nb; ++i) blocks += (int64_t)tiles[i].mcux * tiles[i].mcuy * tiles[i].bpm;
    BQ_CUDA(ctx, cudaMemsetAsync(st, 0, (size_t)nb * 12, ctx->stream));
    BQ_CUDA(ctx, cudaMemsetAsync(coef.p, 0, (size_t)blocks * 128, ctx->stream));
    J::jpeg_unstuff_kernel<<<nb, J::kUnstuffThreads, 0, ctx->stream>>>(d, src, (uint8_t*)ub.p, (int32_t*)intv.p, status);
    BQ_LAUNCH_CHECK(ctx);
    J::jpeg_huffman_kernel<<<nb, J::kHuffThreads, 0, ctx->stream>>>(d, (const uint8_t*)ub.p, (const int32_t*)intv.p,
                                                                    (int32_t*)ichunk.p, (J::Chunk*)chunks.p,
                                                                    (int16_t*)coef.p, status, st);
    BQ_LAUNCH_CHECK(ctx);
    // this call's decode options (prepare sets them on every call) pick the instantiation; the grids do not depend on them
    const dim3 gi((unsigned)((max_tile_blocks + J::kIdctBlocks - 1) / J::kIdctBlocks), (unsigned)nb);
    const auto idct = flags & BQ_JPEG_IDCT_IFAST ? J::jpeg_idct_kernel<J::Idct::kIfast>
                                                 : J::jpeg_idct_kernel<J::Idct::kIslow>;
    idct<<<gi, J::kIdctThreads, 0, ctx->stream>>>(d, (const int16_t*)coef.p, status, (uint8_t*)planes.p, pitch);
    BQ_LAUNCH_CHECK(ctx);
    const dim3 gc((unsigned)((px * px + 255) / 256), (unsigned)nb);
    const auto color = flags & BQ_JPEG_REPLICATE_CHROMA ? J::jpeg_color_kernel<J::Upsample::kReplicate>
                                                        : J::jpeg_color_kernel<J::Upsample::kFancy>;
    color<<<gc, 256, 0, ctx->stream>>>(d, (const uint8_t*)planes.p, status, pitch, px, out);
    BQ_LAUNCH_CHECK(ctx);
    return BQ_OK;
  }

  // subsequence statistics of the whole call, for bq_jpeg_last_stats
  int finished(bq_ctx* ctx) override {
    std::vector<int32_t> s((size_t)n * 3);
    BQ_CUDA(ctx, cudaMemcpy(s.data(), stats.p, s.size() * 4, cudaMemcpyDeviceToHost));
    last_stats[0] = n;
    last_stats[1] = last_stats[2] = last_stats[3] = 0;
    for (int64_t i = 0; i < n; ++i) {
      last_stats[1] += s[3 * i];
      last_stats[2] = std::max<int64_t>(last_stats[2], s[3 * i + 1]);
      last_stats[3] += s[3 * i + 2];
    }
    return BQ_OK;
  }
};

}  // namespace

bq_encoded* bq_jpeg_state(bq_encoded*& slot) { return slot ? slot : (slot = new Jpeg()); }

extern "C" {

const char* bq_jpeg_status_string(int32_t status) { return status_string(status); }

int bq_jpeg_inspect(const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, int32_t* status) {
  return bq_encoded_inspect(Jpeg(), data, offsets, n, px, status);
}

int bq_jpeg_decode(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, uint8_t* out_u8,
                   int32_t* status) {
  return bq_jpeg_decode_ex(ctx, data, offsets, n, px, 0, out_u8, status);
}

int bq_jpeg_decode_ex(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, int32_t flags,
                      uint8_t* out_u8, int32_t* status) {
  return ctx ? bq_encoded_decode(ctx, bq_jpeg_state(ctx->jpeg), data, offsets, n, px, flags, out_u8, status)
             : BQ_ERR_ARG;
}

int bq_jpeg_last_stats(bq_ctx* ctx, int64_t stats[4]) {
  if (!ctx || !stats) return BQ_ERR_ARG;
  for (int k = 0; k < 4; ++k) stats[k] = ctx->jpeg ? static_cast<const Jpeg*>(ctx->jpeg)->last_stats[k] : 0;
  return BQ_OK;
}

}  // extern "C"
