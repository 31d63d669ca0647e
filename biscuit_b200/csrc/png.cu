// PNG tiles on the GPU: the host chunk parse into per-tile descriptors, the layout of their decode scratch and the
// three decode launches of png_sm100.cuh, driven by encoded.cu, and the bq_png_* entry points.
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "../../include/biscuit_b200.h"
#include "encoded.cuh"
#include "png_sm100.cuh"

using bq::png::Tile;

namespace {

const uint8_t kSignature[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};

uint32_t crc32(const uint8_t* p, int64_t n) {
  static const std::vector<uint32_t> table = [] {
    std::vector<uint32_t> t(256);
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (c & 1 ? 0xEDB88320u : 0u);
      t[i] = c;
    }
    return t;
  }();
  uint32_t c = 0xFFFFFFFFu;
  for (int64_t i = 0; i < n; ++i) c = table[(c ^ p[i]) & 255] ^ (c >> 8);
  return c ^ 0xFFFFFFFFu;
}

uint32_t be32(const uint8_t* p) { return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3]; }

bool is_type(const uint8_t* p, const char* t) { return memcmp(p, t, 4) == 0; }

// Chunk parse of one file b[0, len) of which the first `avail` bytes are at hand.  Returns BQ_PNG_* (t.idat filled on
// BQ_PNG_OK) or bq_encoded::kNeedMore.
int parse_tile(const uint8_t* b, int64_t len, int64_t avail, int px, Tile& t) {
  memset(&t, 0, sizeof(t));
#define NEED(k)                                                  \
  do {                                                           \
    if ((int64_t)(k) > len) return BQ_PNG_TRUNCATED_HEADER;      \
    if ((int64_t)(k) > avail) return bq_encoded::kNeedMore;      \
  } while (0)
  if (memcmp(b, kSignature, (size_t)std::min<int64_t>(len, 8)) != 0) return BQ_PNG_NOT_PNG;
  NEED(8);
  bool ihdr = false;
  int64_t i = 8;
  for (;;) {
    NEED(i + 8);
    const int64_t L = be32(b + i);
    const uint8_t* type = b + i + 4;
    if (!ihdr && (!is_type(type, "IHDR") || L != 13)) return BQ_PNG_BAD_IHDR;   // IHDR comes first
    if (is_type(type, "IDAT")) {
      t.idat = (int32_t)i;
      // the two-byte zlib header, possibly spread over several IDAT chunks
      uint8_t z[2];
      int got = 0;
      for (int64_t q = i; got < 2;) {
        NEED(q + 8);
        if (!is_type(b + q + 4, "IDAT")) return BQ_PNG_BAD_ZLIB;
        const int64_t Lq = be32(b + q);
        for (int64_t k = 0; k < Lq && got < 2; ++k) {
          NEED(q + 9 + k);
          z[got++] = b[q + 8 + k];
        }
        q += 12 + Lq;
      }
      if ((z[0] & 15) != 8 || (z[0] >> 4) > 7 || ((int)z[0] << 8 | z[1]) % 31 != 0) return BQ_PNG_BAD_ZLIB;
      if (z[1] & 0x20) return BQ_PNG_PRESET_DICT;
      return BQ_PNG_OK;
    }
    NEED(i + 12 + L);
    if (crc32(b + i + 4, L + 4) != be32(b + i + 8 + L)) return BQ_PNG_BAD_CRC;
    const uint8_t* d = b + i + 8;
    if (is_type(type, "IHDR")) {
      if (ihdr) return BQ_PNG_BAD_IHDR;
      ihdr = true;
      const uint32_t w = be32(d), h = be32(d + 4);
      const int depth = d[8], ct = d[9];
      if (w == 0 || h == 0 || d[10] != 0 || d[11] != 0 || d[12] > 1) return BQ_PNG_BAD_IHDR;
      if (ct == 0 || ct == 3 || ct == 4 || ct == 6) return BQ_PNG_COLOUR_TYPE;
      if (ct != 2) return BQ_PNG_BAD_IHDR;
      if (depth != 8) return BQ_PNG_BIT_DEPTH;
      if (d[12] == 1) return BQ_PNG_INTERLACED;
      if (w != (uint32_t)px || h != (uint32_t)px) return BQ_PNG_SIZE;
    } else if (is_type(type, "IEND")) {
      return BQ_PNG_NO_IDAT;
    } else if (!(type[0] & 0x20) && !is_type(type, "PLTE")) {
      return BQ_PNG_UNKNOWN_CRITICAL;                   // ancillary chunks (lower-case first letter) and PLTE are skipped
    }
    i += 12 + L;
  }
#undef NEED
}

const char* status_string(int32_t s) {
  switch (s) {
    case BQ_PNG_OK: return "ok";
    case BQ_PNG_NOT_PNG: return "not a PNG file (no PNG signature)";
    case BQ_PNG_TRUNCATED_HEADER: return "truncated header: the file ends before its first IDAT chunk and zlib header";
    case BQ_PNG_BAD_CRC: return "bad chunk CRC in a chunk before the image data";
    case BQ_PNG_BAD_IHDR: return "bad IHDR (missing, not first, wrong length, or invalid fields)";
    case BQ_PNG_SIZE: return "image size differs from the model's tile size";
    case BQ_PNG_BIT_DEPTH: return "bit depth is not 8";
    case BQ_PNG_COLOUR_TYPE: return "colour type is not RGB (grayscale / palette / alpha PNG is not supported)";
    case BQ_PNG_INTERLACED: return "interlaced (Adam7) PNG is not supported";
    case BQ_PNG_UNKNOWN_CRITICAL: return "unknown critical chunk";
    case BQ_PNG_NO_IDAT: return "no IDAT chunk before IEND";
    case BQ_PNG_BAD_ZLIB: return "bad zlib header (compression method 8, window <= 32 KB and a valid check expected)";
    case BQ_PNG_PRESET_DICT: return "zlib stream needs a preset dictionary";
    case BQ_PNG_TRUNCATED_DATA: return "truncated data (the IDAT run or the DEFLATE stream ends early, or no Adler-32)";
    case BQ_PNG_BAD_BLOCK: return "bad block (DEFLATE block type 3, or a stored block whose LEN != ~NLEN)";
    case BQ_PNG_BAD_HUFFMAN: return "bad Huffman code (invalid code lengths or an invalid symbol)";
    case BQ_PNG_BAD_DISTANCE: return "bad distance (a match reaches before the start of the stream)";
    case BQ_PNG_WRONG_SIZE: return "wrong decompressed size (not height x (1 + 3 x width) bytes)";
    case BQ_PNG_ADLER: return "Adler-32 mismatch";
    case BQ_PNG_BAD_FILTER: return "bad filter type (a row's filter byte is > 4)";
    default: return "unknown status";
  }
}

int raw_bytes(int px) { return px * (1 + 3 * px); }

// Decode state of one caller: the driver's, plus the PNG decode scratch sized for the largest group.
struct Png final : bq_encoded {
  DevBuf zbuf, zlen, filt, adler;

  const char* name() const override { return "PNG"; }
  size_t desc_bytes() const override { return sizeof(Tile); }
  int head_bytes() const override { return 1024; }
  bool px_ok(int px) const override { return px >= 1 && bq::png::unfilter_smem(px) <= 227 * 1024; }
  int64_t max_tile_bytes() const override { return INT32_MAX; }
  int parse(const uint8_t* b, int64_t len, int64_t avail, const uint8_t*, int px, void* desc) const override {
    return parse_tile(b, len, avail, px, *(Tile*)desc);
  }
  const char* status_string(int32_t code) const override { return ::status_string(code); }

  // tile offsets relative to the group
  int layout(bq_ctx* ctx) override {
    Tile* tiles = (Tile*)desc_host;
    for (int64_t g = 0; g < n_groups(); ++g)
      for (int64_t i = g * group; i < group_end(g); ++i) {
        tiles[i].off = offs[i] - offs[g * group];
        tiles[i].len = (int32_t)(offs[i + 1] - offs[i]);
      }
    const int64_t gmax = std::min(n, group);
    int rc;
    if ((rc = bq_alloc(ctx, zbuf, max_bytes + 16)) || (rc = bq_alloc(ctx, zlen, (size_t)gmax * 4)) ||
        (rc = bq_alloc(ctx, filt, (size_t)gmax * raw_bytes(px))) || (rc = bq_alloc(ctx, adler, (size_t)gmax * 4)))
      return rc;
    return BQ_OK;
  }

  int launch(bq_ctx* ctx, int64_t, int nb, const uint8_t* src, const void* desc_dev, int32_t* status,
             uint8_t* out) override {
    namespace P = bq::png;
    const Tile* d = (const Tile*)desc_dev;
    P::png_dechunk_kernel<<<nb, P::kDechunkThreads, 0, ctx->stream>>>(d, src, (uint8_t*)zbuf.p, (int32_t*)zlen.p,
                                                                      status);
    BQ_LAUNCH_CHECK(ctx);
    P::png_inflate_kernel<<<(nb + P::kInflateWarps - 1) / P::kInflateWarps, 32 * P::kInflateWarps, 0, ctx->stream>>>(
        d, (const uint8_t*)zbuf.p, (const int32_t*)zlen.p, nb, raw_bytes(px), (uint8_t*)filt.p, (uint32_t*)adler.p,
        status);
    BQ_LAUNCH_CHECK(ctx);
    const size_t smem = P::unfilter_smem(px);
    if (smem > 48 * 1024)
      BQ_CUDA(ctx, cudaFuncSetAttribute(P::png_unfilter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    P::png_unfilter_kernel<<<nb, 32, smem, ctx->stream>>>((const uint8_t*)filt.p, px, (const uint32_t*)adler.p, status,
                                                          out);
    BQ_LAUNCH_CHECK(ctx);
    return BQ_OK;
  }
};

}  // namespace

bq_encoded* bq_png_state(bq_encoded*& slot) { return slot ? slot : (slot = new Png()); }

extern "C" {

const char* bq_png_status_string(int32_t status) { return status_string(status); }

int bq_png_inspect(const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, int32_t* status) {
  return bq_encoded_inspect(Png(), data, offsets, n, px, status);
}

int bq_png_decode(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, uint8_t* out_u8,
                  int32_t* status) {
  return ctx ? bq_encoded_decode(ctx, bq_png_state(ctx->png), data, offsets, n, px, 0, out_u8, status) : BQ_ERR_ARG;
}

}  // extern "C"
