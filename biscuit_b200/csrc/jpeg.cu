// Baseline-JPEG tiles on the GPU: host marker parse -> per-tile descriptors, staging, the four decode launches of
// jpeg_sm100.cuh, and the bq_jpeg_* entry points.  bq_predict_uq_jpeg (model.cu) drives the same state per micro-batch.
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "../../include/biscuit_b200.h"
#include "common.cuh"
#include "jpeg_sm100.cuh"

using bq::jpeg::Tile;

namespace {

const uint8_t kNaturalHost[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                  35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                  58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

constexpr int kNeedMore = -1;

// Marker parse of one file b[0, len) of which the first `avail` bytes are at hand (tail2 = its last two bytes).
// Returns BQ_JPEG_* (t filled on BQ_JPEG_OK; t.seg_off relative to the file start) or kNeedMore.
int parse_tile(const uint8_t* b, int64_t len, int64_t avail, const uint8_t* tail2, int px, Tile& t) {
  memset(&t, 0, sizeof(t));
#define NEED(k)                                        \
  do {                                                 \
    if ((int64_t)(k) > len) return BQ_JPEG_TRUNCATED_HEADER; \
    if ((int64_t)(k) > avail) return kNeedMore;        \
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

}  // namespace

// Decode state of one caller (the ctx's bq_jpeg_decode, or one model's bq_predict_uq_jpeg): descriptors of all tiles,
// split into groups of at most `group` tiles that are staged and decoded one at a time; device scratch sized for the
// largest group (grown on demand, never shrunk).
struct bq_jpeg_state {
  const uint8_t* data = nullptr;
  bool on_dev = false;
  int px = 0;
  int64_t n = 0, group = 0;
  std::vector<int64_t> offs;
  Tile* desc_host = nullptr;           // pinned [n]
  size_t desc_host_cap = 0;
  DevBuf stage[2], desc[2];            // compressed bytes / descriptors of a group (double-buffered)
  DevBuf ub, intv, ichunk, chunks, coef, planes, status, stats, heads, offs_dev;
  size_t max_bytes = 0;
  int64_t max_int = 0, max_chunks = 0, max_blocks = 0, max_tile_blocks = 0;
  int64_t last_stats[4] = {};
  ~bq_jpeg_state() { if (desc_host) cudaFreeHost(desc_host); }
};

void bq_jpeg_state_destroy(bq_jpeg_state* s) { delete s; }

static int64_t n_groups(const bq_jpeg_state* s) { return (s->n + s->group - 1) / s->group; }

// Parse every tile (nothing is launched when one is rejected), lay out the groups and size the scratch.
int bq_jpeg_prepare(bq_ctx* ctx, bq_jpeg_state*& s, const uint8_t* data, const int64_t* offsets, int64_t n, int px,
                    int64_t group, int32_t* status_host) {
  if (!s) s = new bq_jpeg_state();
  if (n < 0 || px < 16 || px > 4096 || group < 1 || (n > 0 && (!data || !offsets)))
    return bq_fail(ctx, BQ_ERR_ARG, "bq_jpeg: bad argument");
  for (int64_t i = 0; i < n; ++i)
    if (offsets[i] < 0 || offsets[i + 1] < offsets[i])
      return bq_fail(ctx, BQ_ERR_ARG, "bq_jpeg: offsets must be non-negative and non-decreasing (tile %lld)", (long long)i);
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
      const uint8_t* b = data + offsets[i];
      const uint8_t tail[2] = {len >= 2 ? b[len - 2] : (uint8_t)0, len >= 1 ? b[len - 1] : (uint8_t)0};
      st[i] = parse_tile(b, len, len, tail, px, s->desc_host[i]);
    }
  } else if (n > 0) {
    // device bytes: fetch each tile's first kHead bytes and last two; parse again from the whole tile when the headers
    // run past kHead (large APPn segments)
    constexpr int kHead = 2048;
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
      const uint8_t* h = heads.data() + (size_t)i * (kHead + 2);
      st[i] = parse_tile(h, len, std::min<int64_t>(len, kHead), h + kHead, px, s->desc_host[i]);
      if (st[i] == kNeedMore) {
        whole.resize((size_t)len);
        BQ_CUDA(ctx, cudaMemcpy(whole.data(), data + offsets[i], (size_t)len, cudaMemcpyDeviceToHost));
        st[i] = parse_tile(whole.data(), len, len, h + kHead, px, s->desc_host[i]);
      }
    }
  }
  if (status_host) memcpy(status_host, st.data(), (size_t)n * 4);
  for (int64_t i = 0; i < n; ++i)
    if (st[i] != BQ_JPEG_OK)
      return bq_fail(ctx, BQ_ERR_DATA, "JPEG tile %lld: %s", (long long)i, status_string(st[i]));
  // group layout: every base is relative to the group
  s->max_bytes = 0;
  s->max_int = s->max_chunks = s->max_blocks = s->max_tile_blocks = 0;
  for (int64_t g = 0; g < n_groups(s); ++g) {
    const int64_t i0 = g * group, i1 = std::min(n, i0 + group);
    int64_t ni = 0, nc = 0, nbk = 0;
    for (int64_t i = i0; i < i1; ++i) {
      Tile& t = s->desc_host[i];
      t.seg_off += offsets[i] - offsets[i0];
      t.int_base = (int32_t)ni;
      t.chunk_base = (int32_t)nc;
      t.coef_base = nbk;
      const int64_t blocks = (int64_t)t.mcux * t.mcuy * t.bpm;
      ni += t.n_int + 1;
      nc += t.chunk_cap;
      nbk += blocks;
      s->max_tile_blocks = std::max(s->max_tile_blocks, blocks);
    }
    if (nc > INT32_MAX || ni > INT32_MAX) return bq_fail(ctx, BQ_ERR_ARG, "bq_jpeg: group too large");
    s->max_bytes = std::max(s->max_bytes, (size_t)(offsets[i1] - offsets[i0]));
    s->max_int = std::max(s->max_int, ni);
    s->max_chunks = std::max(s->max_chunks, nc);
    s->max_blocks = std::max(s->max_blocks, nbk);
  }
  const size_t pitch = bq_align_up((size_t)px, 16);
  const int64_t gmax = std::min(n, group);
  int rc;
  if ((!s->on_dev && ((rc = bq_alloc(ctx, s->stage[0], s->max_bytes + 16)) || (rc = bq_alloc(ctx, s->stage[1], s->max_bytes + 16)))) ||
      (rc = bq_alloc(ctx, s->desc[0], (size_t)gmax * sizeof(Tile))) || (rc = bq_alloc(ctx, s->desc[1], (size_t)gmax * sizeof(Tile))) ||
      (rc = bq_alloc(ctx, s->ub, s->max_bytes + 16)) || (rc = bq_alloc(ctx, s->intv, (size_t)s->max_int * 4)) ||
      (rc = bq_alloc(ctx, s->ichunk, (size_t)s->max_int * 4)) ||
      (rc = bq_alloc(ctx, s->chunks, (size_t)s->max_chunks * sizeof(bq::jpeg::Chunk))) ||
      (rc = bq_alloc(ctx, s->coef, (size_t)s->max_blocks * 128)) ||
      (rc = bq_alloc(ctx, s->planes, (size_t)gmax * 3 * pitch * pitch)) ||
      (rc = bq_alloc(ctx, s->status, (size_t)std::max<int64_t>(n, 1) * 4)) ||
      (rc = bq_alloc(ctx, s->stats, (size_t)std::max<int64_t>(n, 1) * 12)))
    return rc;
  return BQ_OK;
}

int64_t bq_jpeg_group_count(const bq_jpeg_state* s) { return n_groups(s); }

int bq_gather_heads(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets_dev, int64_t n, int head, uint8_t* out) {
  bq::jpeg::jpeg_gather_heads_kernel<<<(unsigned)n, 256, 0, ctx->stream>>>(data, offsets_dev, head, out);
  BQ_LAUNCH_CHECK(ctx);
  return BQ_OK;
}

// Copy group g's descriptors (and its bytes, when they are in host memory) into slot `slot` on `stream`.
int bq_jpeg_upload(bq_ctx* ctx, bq_jpeg_state* s, int64_t g, int slot, cudaStream_t stream) {
  const int64_t i0 = g * s->group, i1 = std::min(s->n, i0 + s->group);
  BQ_CUDA(ctx, cudaMemcpyAsync(s->desc[slot].p, s->desc_host + i0, (size_t)(i1 - i0) * sizeof(Tile),
                               cudaMemcpyHostToDevice, stream));
  if (!s->on_dev)
    BQ_CUDA(ctx, cudaMemcpyAsync(s->stage[slot].p, s->data + s->offs[i0], (size_t)(s->offs[i1] - s->offs[i0]),
                                 cudaMemcpyHostToDevice, stream));
  return BQ_OK;
}

// Decode group g (uploaded into `slot`) on the ctx stream into out = uint8 NHWC [group tiles, px, px, 3] (device).
int bq_jpeg_decode_group(bq_ctx* ctx, bq_jpeg_state* s, int64_t g, int slot, uint8_t* out) {
  namespace J = bq::jpeg;
  const int64_t i0 = g * s->group, i1 = std::min(s->n, i0 + s->group);
  const int nb = (int)(i1 - i0);
  const int px = s->px, pitch = (int)bq_align_up((size_t)px, 16);
  const uint8_t* src = s->on_dev ? s->data + s->offs[i0] : (const uint8_t*)s->stage[slot].p;
  const Tile* d = (const Tile*)s->desc[slot].p;
  int32_t* status = (int32_t*)s->status.p + i0;
  int32_t* stats = (int32_t*)s->stats.p + 3 * i0;
  int64_t blocks = 0;
  for (int64_t i = i0; i < i1; ++i) blocks += (int64_t)s->desc_host[i].mcux * s->desc_host[i].mcuy * s->desc_host[i].bpm;
  BQ_CUDA(ctx, cudaMemsetAsync(status, 0, (size_t)nb * 4, ctx->stream));
  BQ_CUDA(ctx, cudaMemsetAsync(stats, 0, (size_t)nb * 12, ctx->stream));
  BQ_CUDA(ctx, cudaMemsetAsync(s->coef.p, 0, (size_t)blocks * 128, ctx->stream));
  J::jpeg_unstuff_kernel<<<nb, J::kUnstuffThreads, 0, ctx->stream>>>(d, src, (uint8_t*)s->ub.p, (int32_t*)s->intv.p, status);
  BQ_LAUNCH_CHECK(ctx);
  J::jpeg_huffman_kernel<<<nb, J::kHuffThreads, 0, ctx->stream>>>(d, (const uint8_t*)s->ub.p, (const int32_t*)s->intv.p,
                                                                  (int32_t*)s->ichunk.p, (J::Chunk*)s->chunks.p,
                                                                  (int16_t*)s->coef.p, status, stats);
  BQ_LAUNCH_CHECK(ctx);
  const dim3 gi((unsigned)((s->max_tile_blocks + J::kIdctBlocks - 1) / J::kIdctBlocks), (unsigned)nb);
  J::jpeg_idct_kernel<<<gi, J::kIdctThreads, 0, ctx->stream>>>(d, (const int16_t*)s->coef.p, status, (uint8_t*)s->planes.p,
                                                               pitch);
  BQ_LAUNCH_CHECK(ctx);
  const dim3 gc((unsigned)((px * px + 255) / 256), (unsigned)nb);
  J::jpeg_color_kernel<<<gc, 256, 0, ctx->stream>>>(d, (const uint8_t*)s->planes.p, status, pitch, px, out);
  BQ_LAUNCH_CHECK(ctx);
  return BQ_OK;
}

// After the last group: wait, fetch the per-tile status, and fail with the first rejected tile.
int bq_jpeg_finish(bq_ctx* ctx, bq_jpeg_state* s, int32_t* status_host) {
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (s->n == 0) return BQ_OK;
  std::vector<int32_t> st((size_t)s->n), stats((size_t)s->n * 3);
  BQ_CUDA(ctx, cudaMemcpy(st.data(), s->status.p, st.size() * 4, cudaMemcpyDeviceToHost));
  BQ_CUDA(ctx, cudaMemcpy(stats.data(), s->stats.p, stats.size() * 4, cudaMemcpyDeviceToHost));
  s->last_stats[0] = s->n;
  s->last_stats[1] = s->last_stats[2] = s->last_stats[3] = 0;
  for (int64_t i = 0; i < s->n; ++i) {
    s->last_stats[1] += stats[3 * i];
    s->last_stats[2] = std::max<int64_t>(s->last_stats[2], stats[3 * i + 1]);
    s->last_stats[3] += stats[3 * i + 2];
  }
  if (status_host) memcpy(status_host, st.data(), st.size() * 4);
  for (int64_t i = 0; i < s->n; ++i)
    if (st[i] != BQ_JPEG_OK)
      return bq_fail(ctx, BQ_ERR_DATA, "JPEG tile %lld: %s", (long long)i, status_string(st[i]));
  return BQ_OK;
}

extern "C" {

const char* bq_jpeg_status_string(int32_t status) { return status_string(status); }

int bq_jpeg_inspect(const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, int32_t* status) {
  if (n < 0 || !status || (n > 0 && (!data || !offsets))) return BQ_ERR_ARG;
  for (int64_t i = 0; i < n; ++i) {
    const int64_t len = offsets[i + 1] - offsets[i];
    if (offsets[i] < 0 || len < 0) return BQ_ERR_ARG;
    const uint8_t* b = data + offsets[i];
    const uint8_t tail[2] = {len >= 2 ? b[len - 2] : (uint8_t)0, len >= 1 ? b[len - 1] : (uint8_t)0};
    Tile t;
    status[i] = parse_tile(b, len, len, tail, px, t);
  }
  return BQ_OK;
}

int bq_jpeg_decode(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, uint8_t* out_u8,
                   int32_t* status) {
  if (!ctx) return BQ_ERR_ARG;
  if (n > 0 && !out_u8) return bq_fail(ctx, BQ_ERR_ARG, "bq_jpeg_decode: bad argument");
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  constexpr int64_t kGroup = 512;
  int rc = bq_jpeg_prepare(ctx, ctx->jpeg, data, offsets, n, px, kGroup, status);
  if (rc) return rc;
  bq_jpeg_state* s = ctx->jpeg;
  const size_t tile_bytes = (size_t)px * px * 3;
  const bool out_dev = bq_is_device_ptr(out_u8);
  DevBuf tmp;
  if (!out_dev && n > 0 && (rc = bq_alloc(ctx, tmp, (size_t)std::min(n, kGroup) * tile_bytes))) return rc;
  for (int64_t g = 0; g < n_groups(s); ++g) {
    const int64_t i0 = g * kGroup, nb = std::min(n - i0, kGroup);
    uint8_t* dst = out_dev ? out_u8 + (size_t)i0 * tile_bytes : (uint8_t*)tmp.p;
    if ((rc = bq_jpeg_upload(ctx, s, g, 0, ctx->stream)) || (rc = bq_jpeg_decode_group(ctx, s, g, 0, dst))) return rc;
    if (!out_dev) BQ_CUDA(ctx, cudaMemcpyAsync(out_u8 + (size_t)i0 * tile_bytes, dst, (size_t)nb * tile_bytes,
                                               cudaMemcpyDeviceToHost, ctx->stream));
  }
  rc = bq_jpeg_finish(ctx, s, status);
  if (!out_dev) BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // tmp is released below
  return rc;
}

int bq_jpeg_last_stats(bq_ctx* ctx, int64_t stats[4]) {
  if (!ctx || !stats) return BQ_ERR_ARG;
  for (int k = 0; k < 4; ++k) stats[k] = ctx->jpeg ? ctx->jpeg->last_stats[k] : 0;
  return BQ_OK;
}

}  // extern "C"
