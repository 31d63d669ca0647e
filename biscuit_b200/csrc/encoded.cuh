// Compressed tiles (JPEG, PNG) on the GPU: the driver every format shares.  A format turns each file's headers into a
// fixed-size descriptor on the host and launches its decode kernels; the driver (encoded.cu) checks the arguments,
// parses host or device-resident bytes and names the first rejected tile before anything is launched, stages the tiles
// group by group, and names the first tile the kernels rejected.  bq_{jpeg,png}_decode (jpeg.cu, png.cu) and
// bq_predict_uq_{jpeg,png} (model.cu) drive it.
#pragma once

#include <algorithm>
#include <string>
#include <vector>

#include "common.cuh"

// Decode state of one caller (a ctx's bq_*_decode, or one model's bq_predict_uq_*) for one format: descriptors of all
// tiles, split into groups of at most `group` tiles that are staged and decoded one at a time; device scratch sized for
// the largest group (grown on demand, never shrunk).
struct bq_encoded {
  static constexpr int kNeedMore = -1;  // parse: the headers run past the `avail` bytes at hand

  // ---- the format
  virtual const char* name() const = 0;                        // "JPEG" / "PNG": the prefix of every message
  virtual size_t desc_bytes() const = 0;                       // size of one tile's descriptor
  virtual int head_bytes() const = 0;                          // bytes fetched per device-resident tile for the parse
  virtual bool px_ok(int px) const = 0;                        // tile sizes the kernels decode
  // Longest file the descriptor addresses; INT32_MAX when it holds a length in 32 bits ("tiles < 2 GB").
  virtual int64_t max_tile_bytes() const { return INT64_MAX; }
  // Decode-option bits the format accepts in a call's `flags` (JPEG: BQ_JPEG_IDCT_IFAST | BQ_JPEG_REPLICATE_CHROMA;
  // PNG: BQ_PNG_CONVERT_RGB).
  virtual int32_t known_flags() const { return 0; }
  // Header parse of one file b[0, len) of which the first `avail` bytes are at hand (tail2 = its last two bytes) under
  // the call's decode options `flags`: fills the descriptor `desc` and returns the format's status code (0 =
  // accepted), or kNeedMore.
  virtual int parse(const uint8_t* b, int64_t len, int64_t avail, const uint8_t* tail2, int px, int32_t flags,
                    void* desc) const = 0;
  virtual const char* status_string(int32_t code) const = 0;
  // After a successful parse: rebase every group's descriptors to its group, size and allocate the format's scratch.
  virtual int layout(bq_ctx* ctx) = 0;
  // Decode tiles [i0, i0 + nb), one group, on the ctx stream: their bytes start at src and their descriptors at
  // desc_dev; status (one per tile, zeroed) and out (uint8 NHWC) start at tile i0.
  virtual int launch(bq_ctx* ctx, int64_t i0, int nb, const uint8_t* src, const void* desc_dev, int32_t* status,
                     uint8_t* out) = 0;
  // After the last group, once the stream is idle (n > 0).
  virtual int finished(bq_ctx*) { return BQ_OK; }

  // ---- the driver (encoded.cu)
  // Parse every tile (nothing is launched when one is rejected), lay out the groups and size the scratch.  `flags` are
  // the call's decode options; every call sets them, so none carries over to the next call on the same state.
  int prepare(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int px, int64_t group,
              int32_t flags, int32_t* status_host);
  // Copy group g's descriptors (and its bytes, when they are in host memory) into slot `slot` on `stream`.
  int upload(bq_ctx* ctx, int64_t g, int slot, cudaStream_t stream);
  // Decode group g (uploaded into `slot`) on the ctx stream into out = uint8 NHWC [group tiles, px, px, 3] (device).
  int decode_group(bq_ctx* ctx, int64_t g, int slot, uint8_t* out);
  // After the last group: wait, fetch the per-tile status, and fail with the first rejected tile.
  int finish(bq_ctx* ctx, int32_t* status_host);

  int64_t n_groups() const { return (n + group - 1) / group; }
  int64_t group_end(int64_t g) const { return std::min(n, (g + 1) * group); }
  std::string api() const;                                     // "jpeg" / "png": in entry-point names
  virtual ~bq_encoded() { if (desc_host) cudaFreeHost(desc_host); }

  const uint8_t* data = nullptr;
  bool on_dev = false;
  int px = 0;
  int32_t flags = 0;
  int64_t n = 0, group = 0;
  std::vector<int64_t> offs;
  void* desc_host = nullptr;           // pinned [n] descriptors
  size_t desc_host_cap = 0;
  DevBuf stage[2], desc[2];            // compressed bytes / descriptors of a group (double-buffered)
  DevBuf status, heads, offs_dev;
  size_t max_bytes = 0;                // compressed bytes of the largest group

 private:
  int report(bq_ctx* ctx, const std::vector<int32_t>& st, int32_t* status_host);
};

// Bodies of bq_{jpeg,png}_inspect and bq_{jpeg,png}_decode (ctx != NULL); decode stages groups of 512 tiles.
int bq_encoded_inspect(const bq_encoded& f, const uint8_t* data, const int64_t* offsets, int64_t n, int px,
                       int32_t flags, int32_t* status);
int bq_encoded_decode(bq_ctx* ctx, bq_encoded* s, const uint8_t* data, const int64_t* offsets, int64_t n, int px,
                      int32_t flags, uint8_t* out_u8, int32_t* status);

// The JPEG (jpeg.cu) / PNG (png.cu) state kept in `slot`, created on first use.
bq_encoded* bq_jpeg_state(bq_encoded*& slot);
bq_encoded* bq_png_state(bq_encoded*& slot);
