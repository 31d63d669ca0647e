// PNG tiles on the GPU: host chunk parse -> per-tile descriptors, staging, the three decode launches of png_sm100.cuh,
// and the bq_png_* entry points.  bq_predict_uq_png (model.cu) drives the same state per micro-batch.
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "../../include/biscuit_b200.h"
#include "common.cuh"
#include "png_sm100.cuh"

using bq::png::Tile;

namespace {

constexpr int kNeedMore = -1;
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
// BQ_PNG_OK) or kNeedMore.
int parse_tile(const uint8_t* b, int64_t len, int64_t avail, int px, Tile& t) {
  memset(&t, 0, sizeof(t));
#define NEED(k)                                                  \
  do {                                                           \
    if ((int64_t)(k) > len) return BQ_PNG_TRUNCATED_HEADER;      \
    if ((int64_t)(k) > avail) return kNeedMore;                  \
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

}  // namespace

// Decode state of one caller (the ctx's bq_png_decode, or one model's bq_predict_uq_png): descriptors of all tiles,
// split into groups of at most `group` tiles that are staged and decoded one at a time; device scratch sized for the
// largest group (grown on demand, never shrunk).
struct bq_png_state {
  const uint8_t* data = nullptr;
  bool on_dev = false;
  int px = 0;
  int64_t n = 0, group = 0;
  std::vector<int64_t> offs;
  Tile* desc_host = nullptr;           // pinned [n]
  size_t desc_host_cap = 0;
  DevBuf stage[2], desc[2];            // compressed bytes / descriptors of a group (double-buffered)
  DevBuf zbuf, zlen, filt, adler, status, heads, offs_dev;
  size_t max_bytes = 0;
  ~bq_png_state() { if (desc_host) cudaFreeHost(desc_host); }
};

void bq_png_state_destroy(bq_png_state* s) { delete s; }

static int64_t n_groups(const bq_png_state* s) { return (s->n + s->group - 1) / s->group; }

// Parse every tile (nothing is launched when one is rejected), lay out the groups and size the scratch.
int bq_png_prepare(bq_ctx* ctx, bq_png_state*& s, const uint8_t* data, const int64_t* offsets, int64_t n, int px,
                   int64_t group, int32_t* status_host) {
  if (!s) s = new bq_png_state();
  if (n < 0 || px < 1 || bq::png::unfilter_smem(px) > 227 * 1024 || group < 1 || (n > 0 && (!data || !offsets)))
    return bq_fail(ctx, BQ_ERR_ARG, "bq_png: bad argument");
  for (int64_t i = 0; i < n; ++i)
    if (offsets[i] < 0 || offsets[i + 1] < offsets[i] || offsets[i + 1] - offsets[i] > INT32_MAX)
      return bq_fail(ctx, BQ_ERR_ARG, "bq_png: offsets must be non-negative and non-decreasing, tiles < 2 GB (tile %lld)",
                     (long long)i);
  s->data = data;
  s->on_dev = n > 0 && bq_is_device_ptr(data);
  s->px = px;
  s->n = n;
  s->group = group;
  s->offs.assign(offsets, offsets + n + 1);
  if ((size_t)n > s->desc_host_cap) {
    if (s->desc_host) cudaFreeHost(s->desc_host);
    s->desc_host = nullptr;
    s->desc_host_cap = 0;
    BQ_CUDA(ctx, cudaHostAlloc((void**)&s->desc_host, (size_t)n * sizeof(Tile), cudaHostAllocDefault));
    s->desc_host_cap = (size_t)n;
  }
  std::vector<int32_t> st((size_t)n, 0);
  if (!s->on_dev) {
    for (int64_t i = 0; i < n; ++i) {
      const int64_t len = offsets[i + 1] - offsets[i];
      st[i] = parse_tile(data + offsets[i], len, len, px, s->desc_host[i]);
    }
  } else if (n > 0) {
    // device bytes: fetch each tile's first kHead bytes; parse again from the whole tile when the chunks before the
    // zlib header run past kHead (a large iCCP, for example)
    constexpr int kHead = 1024;
    int rc;
    if ((rc = bq_alloc(ctx, s->offs_dev, (size_t)(n + 1) * 8)) || (rc = bq_alloc(ctx, s->heads, (size_t)n * (kHead + 2))))
      return rc;
    BQ_CUDA(ctx, cudaMemcpyAsync(s->offs_dev.p, offsets, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = bq_gather_heads(ctx, data, (const int64_t*)s->offs_dev.p, n, kHead, (uint8_t*)s->heads.p))) return rc;
    std::vector<uint8_t> heads((size_t)n * (kHead + 2)), whole;
    BQ_CUDA(ctx, cudaMemcpyAsync(heads.data(), s->heads.p, heads.size(), cudaMemcpyDeviceToHost, ctx->stream));
    BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int64_t i = 0; i < n; ++i) {
      const int64_t len = offsets[i + 1] - offsets[i];
      st[i] = parse_tile(heads.data() + (size_t)i * (kHead + 2), len, std::min<int64_t>(len, kHead), px, s->desc_host[i]);
      if (st[i] == kNeedMore) {
        whole.resize((size_t)len);
        BQ_CUDA(ctx, cudaMemcpy(whole.data(), data + offsets[i], (size_t)len, cudaMemcpyDeviceToHost));
        st[i] = parse_tile(whole.data(), len, len, px, s->desc_host[i]);
      }
    }
  }
  if (status_host) memcpy(status_host, st.data(), (size_t)n * 4);
  for (int64_t i = 0; i < n; ++i)
    if (st[i] != BQ_PNG_OK) return bq_fail(ctx, BQ_ERR_DATA, "PNG tile %lld: %s", (long long)i, status_string(st[i]));
  // group layout: tile offsets relative to the group
  s->max_bytes = 0;
  for (int64_t g = 0; g < n_groups(s); ++g) {
    const int64_t i0 = g * group, i1 = std::min(n, i0 + group);
    for (int64_t i = i0; i < i1; ++i) {
      s->desc_host[i].off = offsets[i] - offsets[i0];
      s->desc_host[i].len = (int32_t)(offsets[i + 1] - offsets[i]);
    }
    s->max_bytes = std::max(s->max_bytes, (size_t)(offsets[i1] - offsets[i0]));
  }
  const int64_t gmax = std::min(n, group);
  int rc;
  if ((!s->on_dev && ((rc = bq_alloc(ctx, s->stage[0], s->max_bytes + 16)) || (rc = bq_alloc(ctx, s->stage[1], s->max_bytes + 16)))) ||
      (rc = bq_alloc(ctx, s->desc[0], (size_t)gmax * sizeof(Tile))) || (rc = bq_alloc(ctx, s->desc[1], (size_t)gmax * sizeof(Tile))) ||
      (rc = bq_alloc(ctx, s->zbuf, s->max_bytes + 16)) || (rc = bq_alloc(ctx, s->zlen, (size_t)gmax * 4)) ||
      (rc = bq_alloc(ctx, s->filt, (size_t)gmax * raw_bytes(px))) || (rc = bq_alloc(ctx, s->adler, (size_t)gmax * 4)) ||
      (rc = bq_alloc(ctx, s->status, (size_t)std::max<int64_t>(n, 1) * 4)))
    return rc;
  return BQ_OK;
}

int64_t bq_png_group_count(const bq_png_state* s) { return n_groups(s); }

// Copy group g's descriptors (and its bytes, when they are in host memory) into slot `slot` on `stream`.
int bq_png_upload(bq_ctx* ctx, bq_png_state* s, int64_t g, int slot, cudaStream_t stream) {
  const int64_t i0 = g * s->group, i1 = std::min(s->n, i0 + s->group);
  BQ_CUDA(ctx, cudaMemcpyAsync(s->desc[slot].p, s->desc_host + i0, (size_t)(i1 - i0) * sizeof(Tile),
                               cudaMemcpyHostToDevice, stream));
  if (!s->on_dev)
    BQ_CUDA(ctx, cudaMemcpyAsync(s->stage[slot].p, s->data + s->offs[i0], (size_t)(s->offs[i1] - s->offs[i0]),
                                 cudaMemcpyHostToDevice, stream));
  return BQ_OK;
}

// Decode group g (uploaded into `slot`) on the ctx stream into out = uint8 NHWC [group tiles, px, px, 3] (device).
int bq_png_decode_group(bq_ctx* ctx, bq_png_state* s, int64_t g, int slot, uint8_t* out) {
  namespace P = bq::png;
  const int64_t i0 = g * s->group, i1 = std::min(s->n, i0 + s->group);
  const int nb = (int)(i1 - i0);
  const uint8_t* src = s->on_dev ? s->data + s->offs[i0] : (const uint8_t*)s->stage[slot].p;
  const Tile* d = (const Tile*)s->desc[slot].p;
  int32_t* status = (int32_t*)s->status.p + i0;
  BQ_CUDA(ctx, cudaMemsetAsync(status, 0, (size_t)nb * 4, ctx->stream));
  P::png_dechunk_kernel<<<nb, P::kDechunkThreads, 0, ctx->stream>>>(d, src, (uint8_t*)s->zbuf.p, (int32_t*)s->zlen.p,
                                                                    status);
  BQ_LAUNCH_CHECK(ctx);
  P::png_inflate_kernel<<<(nb + P::kInflateWarps - 1) / P::kInflateWarps, 32 * P::kInflateWarps, 0, ctx->stream>>>(
      d, (const uint8_t*)s->zbuf.p, (const int32_t*)s->zlen.p, nb, raw_bytes(s->px), (uint8_t*)s->filt.p,
      (uint32_t*)s->adler.p, status);
  BQ_LAUNCH_CHECK(ctx);
  const size_t smem = P::unfilter_smem(s->px);
  if (smem > 48 * 1024)
    BQ_CUDA(ctx, cudaFuncSetAttribute(P::png_unfilter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  P::png_unfilter_kernel<<<nb, 32, smem, ctx->stream>>>((const uint8_t*)s->filt.p, s->px, (const uint32_t*)s->adler.p,
                                                        status, out);
  BQ_LAUNCH_CHECK(ctx);
  return BQ_OK;
}

// After the last group: wait, fetch the per-tile status, and fail with the first rejected tile.
int bq_png_finish(bq_ctx* ctx, bq_png_state* s, int32_t* status_host) {
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (s->n == 0) return BQ_OK;
  std::vector<int32_t> st((size_t)s->n);
  BQ_CUDA(ctx, cudaMemcpy(st.data(), s->status.p, st.size() * 4, cudaMemcpyDeviceToHost));
  if (status_host) memcpy(status_host, st.data(), st.size() * 4);
  for (int64_t i = 0; i < s->n; ++i)
    if (st[i] != BQ_PNG_OK) return bq_fail(ctx, BQ_ERR_DATA, "PNG tile %lld: %s", (long long)i, status_string(st[i]));
  return BQ_OK;
}

extern "C" {

const char* bq_png_status_string(int32_t status) { return status_string(status); }

int bq_png_inspect(const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, int32_t* status) {
  if (n < 0 || !status || (n > 0 && (!data || !offsets))) return BQ_ERR_ARG;
  for (int64_t i = 0; i < n; ++i) {
    const int64_t len = offsets[i + 1] - offsets[i];
    if (offsets[i] < 0 || len < 0) return BQ_ERR_ARG;
    Tile t;
    status[i] = parse_tile(data + offsets[i], len, len, px, t);
  }
  return BQ_OK;
}

int bq_png_decode(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, uint8_t* out_u8,
                  int32_t* status) {
  if (!ctx) return BQ_ERR_ARG;
  if (n > 0 && !out_u8) return bq_fail(ctx, BQ_ERR_ARG, "bq_png_decode: bad argument");
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  constexpr int64_t kGroup = 512;
  int rc = bq_png_prepare(ctx, ctx->png, data, offsets, n, px, kGroup, status);
  if (rc) return rc;
  bq_png_state* s = ctx->png;
  const size_t tile_bytes = (size_t)px * px * 3;
  const bool out_dev = bq_is_device_ptr(out_u8);
  DevBuf tmp;
  if (!out_dev && n > 0 && (rc = bq_alloc(ctx, tmp, (size_t)std::min(n, kGroup) * tile_bytes))) return rc;
  for (int64_t g = 0; g < n_groups(s); ++g) {
    const int64_t i0 = g * kGroup, nb = std::min(n - i0, kGroup);
    uint8_t* dst = out_dev ? out_u8 + (size_t)i0 * tile_bytes : (uint8_t*)tmp.p;
    if ((rc = bq_png_upload(ctx, s, g, 0, ctx->stream)) || (rc = bq_png_decode_group(ctx, s, g, 0, dst))) return rc;
    if (!out_dev) BQ_CUDA(ctx, cudaMemcpyAsync(out_u8 + (size_t)i0 * tile_bytes, dst, (size_t)nb * tile_bytes,
                                               cudaMemcpyDeviceToHost, ctx->stream));
  }
  rc = bq_png_finish(ctx, s, status);
  if (!out_dev) BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // tmp is released below
  return rc;
}

}  // extern "C"
