// Shared host-side plumbing of libbiscuit_b200: context, error reporting, device buffers, staging.  The compressed-tile
// states a context keeps per format are declared in encoded.cuh.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/biscuit_b200.h"

struct bq_encoded;      // encoded.cuh

struct bq_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int num_sms = 148;
  int64_t launches = 0;
  std::string err;
  // reusable device scratch (grown on demand, never shrunk)
  void* scratch = nullptr;
  size_t scratch_bytes = 0;
  // small pinned mailbox for scalar results
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
  bq_encoded* jpeg = nullptr;          // bq_jpeg_decode's descriptors and scratch (created on first use)
  bq_encoded* png = nullptr;           // bq_png_decode's, likewise
};

inline int bq_fail(bq_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

#define BQ_CUDA(ctx, expr)                                                                   \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return bq_fail((ctx), BQ_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                     __FILE__, __LINE__);                                                    \
  } while (0)

#define BQ_LAUNCH_CHECK(ctx)                                                                 \
  do {                                                                                       \
    (ctx)->launches++;                                                                       \
    cudaError_t _e = cudaGetLastError();                                                     \
    if (_e != cudaSuccess)                                                                   \
      return bq_fail((ctx), BQ_ERR_CUDA, "kernel launch failed: %s (%s:%d)",                 \
                     cudaGetErrorString(_e), __FILE__, __LINE__);                            \
  } while (0)

inline bool bq_is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Owning or borrowed device array.
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  bool owned = false;
  bool pooled = false;               // allocated with cudaMallocAsync on `stream` (short-lived per-call buffers)
  cudaStream_t stream = nullptr;
  void release() {
    if (owned && p) {
      // stream-ordered free: no device-wide synchronisation (cudaFree costs ~1 ms per buffer with work in flight)
      if (!pooled || cudaFreeAsync(p, stream) != cudaSuccess) { cudaGetLastError(); cudaFree(p); }
    }
    p = nullptr;
    bytes = 0;
    owned = false;
    pooled = false;
  }
  ~DevBuf() { release(); }
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
};

// Make `src` (host or device) available on the device: device pointers are borrowed, host ones copied.
inline int bq_to_device(bq_ctx* ctx, DevBuf& dst, const void* src, size_t bytes) {
  dst.release();
  if (bytes == 0) return BQ_OK;
  if (bq_is_device_ptr(src)) {
    dst.p = const_cast<void*>(src);
    dst.bytes = bytes;
    dst.owned = false;
    return BQ_OK;
  }
  BQ_CUDA(ctx, cudaMalloc(&dst.p, bytes));
  dst.bytes = bytes;
  dst.owned = true;
  BQ_CUDA(ctx, cudaMemcpyAsync(dst.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return BQ_OK;
}

inline int bq_alloc(bq_ctx* ctx, DevBuf& dst, size_t bytes) {
  if (dst.owned && dst.bytes >= bytes) return BQ_OK;
  dst.release();
  if (bytes == 0) return BQ_OK;
  BQ_CUDA(ctx, cudaMalloc(&dst.p, bytes));
  dst.bytes = bytes;
  dst.owned = true;
  return BQ_OK;
}

// Stream-ordered variants for per-call temporaries (thresholding tables, ROC operands): allocation and release are
// queued on the ctx stream and served from the device's default memory pool, whose release threshold bq_create raises
// so the memory stays cached between calls.
inline int bq_alloc_pooled(bq_ctx* ctx, DevBuf& dst, size_t bytes) {
  if (dst.owned && dst.bytes >= bytes) return BQ_OK;
  dst.release();
  if (bytes == 0) return BQ_OK;
  BQ_CUDA(ctx, cudaMallocAsync(&dst.p, bytes, ctx->stream));
  dst.bytes = bytes;
  dst.owned = true;
  dst.pooled = true;
  dst.stream = ctx->stream;
  return BQ_OK;
}

inline int bq_to_device_pooled(bq_ctx* ctx, DevBuf& dst, const void* src, size_t bytes) {
  dst.release();
  if (bytes == 0) return BQ_OK;
  if (bq_is_device_ptr(src)) {
    dst.p = const_cast<void*>(src);
    dst.bytes = bytes;
    dst.owned = false;
    return BQ_OK;
  }
  int rc = bq_alloc_pooled(ctx, dst, bytes);
  if (rc) return rc;
  BQ_CUDA(ctx, cudaMemcpyAsync(dst.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return BQ_OK;
}

// Copy a device result to a caller pointer that may itself be host or device.
inline int bq_from_device(bq_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (!dst || bytes == 0) return BQ_OK;
  BQ_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, ctx->stream));
  return BQ_OK;
}

inline int bq_scratch(bq_ctx* ctx, size_t bytes, void** out) {
  if (ctx->scratch_bytes < bytes) {
    if (ctx->scratch) {
      BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      cudaFree(ctx->scratch);
      ctx->scratch = nullptr;
      ctx->scratch_bytes = 0;
    }
    size_t want = bytes + (bytes >> 2) + 4096;
    BQ_CUDA(ctx, cudaMalloc(&ctx->scratch, want));
    ctx->scratch_bytes = want;
  }
  *out = ctx->scratch;
  return BQ_OK;
}

static inline size_t bq_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
