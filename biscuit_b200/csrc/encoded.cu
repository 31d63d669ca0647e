// The compressed-tile driver (encoded.cuh): argument checks, host / device header parse, group staging, status report,
// and the bodies of the bq_{jpeg,png}_inspect / _decode entry points.
#include <cuda_runtime.h>

#include <cctype>

#include "encoded.cuh"

namespace bq {
namespace encoded {

// Header bytes of tiles resident on the device, for the host header parse: the first `head` bytes of every tile
// (zero-padded) followed by its last two bytes.
__global__ void gather_heads_kernel(const uint8_t* __restrict__ data, const int64_t* __restrict__ offsets, int head,
                                    uint8_t* __restrict__ out) {
  const int64_t i = blockIdx.x;
  const int64_t off = offsets[i], len = offsets[i + 1] - offsets[i];
  uint8_t* o = out + i * (head + 2);
  for (int j = threadIdx.x; j < head + 2; j += blockDim.x) {
    uint8_t v = 0;
    if (j < head) v = j < len ? data[off + j] : 0;
    else if (len >= 2) v = data[off + len - 2 + (j - head)];
    o[j] = v;
  }
}

}  // namespace encoded
}  // namespace bq

namespace {

int parse_host(const bq_encoded& f, const uint8_t* b, int64_t len, int px, int32_t flags, void* desc) {
  const uint8_t tail[2] = {len >= 2 ? b[len - 2] : (uint8_t)0, len >= 1 ? b[len - 1] : (uint8_t)0};
  return f.parse(b, len, len, tail, px, flags, desc);
}

}  // namespace

std::string bq_encoded::api() const {
  std::string s;
  for (const char* c = name(); *c; ++c) s += (char)tolower(*c);
  return s;
}

int bq_encoded::report(bq_ctx* ctx, const std::vector<int32_t>& st, int32_t* status_host) {
  if (status_host) memcpy(status_host, st.data(), st.size() * 4);
  for (size_t i = 0; i < st.size(); ++i)
    if (st[i] != 0) return bq_fail(ctx, BQ_ERR_DATA, "%s tile %lld: %s", name(), (long long)i, status_string(st[i]));
  return BQ_OK;
}

int bq_encoded::prepare(bq_ctx* ctx, const uint8_t* data_, const int64_t* offsets, int64_t n_, int px_, int64_t group_,
                        int32_t flags_, int32_t* status_host) {
  if (n_ < 0 || !px_ok(px_) || group_ < 1 || (n_ > 0 && (!data_ || !offsets)))
    return bq_fail(ctx, BQ_ERR_ARG, "bq_%s: bad argument", api().c_str());
  if (flags_ & ~known_flags())
    return bq_fail(ctx, BQ_ERR_ARG, "bq_%s: unknown decode flag bits 0x%x (known: 0x%x)", api().c_str(),
                   (unsigned)(flags_ & ~known_flags()), (unsigned)known_flags());
  const int64_t cap = max_tile_bytes();
  for (int64_t i = 0; i < n_; ++i)
    if (offsets[i] < 0 || offsets[i + 1] < offsets[i] || offsets[i + 1] - offsets[i] > cap)
      return bq_fail(ctx, BQ_ERR_ARG, "bq_%s: offsets must be non-negative and non-decreasing%s (tile %lld)",
                     api().c_str(), cap < INT64_MAX ? ", tiles < 2 GB" : "", (long long)i);
  data = data_;
  on_dev = n_ > 0 && bq_is_device_ptr(data_);
  px = px_;
  flags = flags_;
  n = n_;
  group = group_;
  offs.assign(offsets, offsets + n + 1);
  const size_t db = desc_bytes();
  if ((size_t)n > desc_host_cap) {
    if (desc_host) cudaFreeHost(desc_host);
    desc_host = nullptr;
    desc_host_cap = 0;
    BQ_CUDA(ctx, cudaHostAlloc(&desc_host, (size_t)n * db, cudaHostAllocDefault));
    desc_host_cap = (size_t)n;
  }
  uint8_t* d = (uint8_t*)desc_host;
  std::vector<int32_t> st((size_t)n, 0);
  if (!on_dev) {
    for (int64_t i = 0; i < n; ++i)
      st[i] = parse_host(*this, data + offsets[i], offsets[i + 1] - offsets[i], px, flags, d + i * db);
  } else if (n > 0) {
    // device bytes: fetch each tile's first `head` bytes and last two; parse again from the whole tile when the headers
    // run past the head (large APPn segments, a large iCCP chunk)
    const int head = head_bytes();
    int rc;
    if ((rc = bq_alloc(ctx, offs_dev, (size_t)(n + 1) * 8)) || (rc = bq_alloc(ctx, heads, (size_t)n * (head + 2))))
      return rc;
    BQ_CUDA(ctx, cudaMemcpyAsync(offs_dev.p, offsets, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    bq::encoded::gather_heads_kernel<<<(unsigned)n, 256, 0, ctx->stream>>>(data, (const int64_t*)offs_dev.p, head,
                                                                           (uint8_t*)heads.p);
    BQ_LAUNCH_CHECK(ctx);
    std::vector<uint8_t> h_all((size_t)n * (head + 2)), whole;
    BQ_CUDA(ctx, cudaMemcpyAsync(h_all.data(), heads.p, h_all.size(), cudaMemcpyDeviceToHost, ctx->stream));
    BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int64_t i = 0; i < n; ++i) {
      const int64_t len = offsets[i + 1] - offsets[i];
      const uint8_t* h = h_all.data() + (size_t)i * (head + 2);
      st[i] = parse(h, len, std::min<int64_t>(len, head), h + head, px, flags, d + i * db);
      if (st[i] == kNeedMore) {
        whole.resize((size_t)len);
        BQ_CUDA(ctx, cudaMemcpy(whole.data(), data + offsets[i], (size_t)len, cudaMemcpyDeviceToHost));
        st[i] = parse(whole.data(), len, len, h + head, px, flags, d + i * db);
      }
    }
  }
  int rc = report(ctx, st, status_host);
  if (rc) return rc;
  max_bytes = 0;
  for (int64_t g = 0; g < n_groups(); ++g)
    max_bytes = std::max(max_bytes, (size_t)(offs[group_end(g)] - offs[g * group]));
  const size_t gmax = (size_t)std::min(n, group);
  if ((!on_dev && ((rc = bq_alloc(ctx, stage[0], max_bytes + 16)) || (rc = bq_alloc(ctx, stage[1], max_bytes + 16)))) ||
      (rc = bq_alloc(ctx, desc[0], gmax * db)) || (rc = bq_alloc(ctx, desc[1], gmax * db)) ||
      (rc = bq_alloc(ctx, status, (size_t)std::max<int64_t>(n, 1) * 4)))
    return rc;
  return layout(ctx);
}

int bq_encoded::upload(bq_ctx* ctx, int64_t g, int slot, cudaStream_t stream) {
  const int64_t i0 = g * group, i1 = group_end(g);
  const size_t db = desc_bytes();
  BQ_CUDA(ctx, cudaMemcpyAsync(desc[slot].p, (const uint8_t*)desc_host + i0 * db, (size_t)(i1 - i0) * db,
                               cudaMemcpyHostToDevice, stream));
  if (!on_dev)
    BQ_CUDA(ctx, cudaMemcpyAsync(stage[slot].p, data + offs[i0], (size_t)(offs[i1] - offs[i0]), cudaMemcpyHostToDevice,
                                 stream));
  return BQ_OK;
}

int bq_encoded::decode_group(bq_ctx* ctx, int64_t g, int slot, uint8_t* out) {
  const int64_t i0 = g * group;
  const int nb = (int)(group_end(g) - i0);
  const uint8_t* src = on_dev ? data + offs[i0] : (const uint8_t*)stage[slot].p;
  int32_t* st = (int32_t*)status.p + i0;
  BQ_CUDA(ctx, cudaMemsetAsync(st, 0, (size_t)nb * 4, ctx->stream));
  return launch(ctx, i0, nb, src, desc[slot].p, st, out);
}

int bq_encoded::finish(bq_ctx* ctx, int32_t* status_host) {
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n == 0) return BQ_OK;
  std::vector<int32_t> st((size_t)n);
  BQ_CUDA(ctx, cudaMemcpy(st.data(), status.p, st.size() * 4, cudaMemcpyDeviceToHost));
  int rc = finished(ctx);
  return rc ? rc : report(ctx, st, status_host);
}

int bq_encoded_inspect(const bq_encoded& f, const uint8_t* data, const int64_t* offsets, int64_t n, int px,
                       int32_t flags, int32_t* status) {
  if (n < 0 || !status || (n > 0 && (!data || !offsets)) || (flags & ~f.known_flags())) return BQ_ERR_ARG;
  std::vector<uint8_t> desc(f.desc_bytes());
  for (int64_t i = 0; i < n; ++i) {
    const int64_t len = offsets[i + 1] - offsets[i];
    if (offsets[i] < 0 || len < 0) return BQ_ERR_ARG;
    status[i] = parse_host(f, data + offsets[i], len, px, flags, desc.data());
  }
  return BQ_OK;
}

int bq_encoded_decode(bq_ctx* ctx, bq_encoded* s, const uint8_t* data, const int64_t* offsets, int64_t n, int px,
                      int32_t flags, uint8_t* out_u8, int32_t* status) {
  if (n > 0 && !out_u8) return bq_fail(ctx, BQ_ERR_ARG, "bq_%s_decode: bad argument", s->api().c_str());
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  constexpr int64_t kGroup = 512;
  int rc = s->prepare(ctx, data, offsets, n, px, kGroup, flags, status);
  if (rc) return rc;
  const size_t tile_bytes = (size_t)px * px * 3;
  const bool out_dev = bq_is_device_ptr(out_u8);
  DevBuf tmp;
  if (!out_dev && n > 0 && (rc = bq_alloc(ctx, tmp, (size_t)std::min(n, kGroup) * tile_bytes))) return rc;
  for (int64_t g = 0; g < s->n_groups(); ++g) {
    const int64_t i0 = g * kGroup, nb = std::min(n - i0, kGroup);
    uint8_t* dst = out_dev ? out_u8 + (size_t)i0 * tile_bytes : (uint8_t*)tmp.p;
    if ((rc = s->upload(ctx, g, 0, ctx->stream)) || (rc = s->decode_group(ctx, g, 0, dst))) return rc;
    if (!out_dev) BQ_CUDA(ctx, cudaMemcpyAsync(out_u8 + (size_t)i0 * tile_bytes, dst, (size_t)nb * tile_bytes,
                                               cudaMemcpyDeviceToHost, ctx->stream));
  }
  rc = s->finish(ctx, status);
  if (!out_dev) BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // tmp is released below
  return rc;
}
