// Bandwidth-bound layers of the Xception-UQ path (NHWC, bf16 storage, fp32 math), coalesced 16-byte accesses:
//   tile_stats  -- per-tile mean / 1/std over the uint8 tile (tf.image.per_image_standardization, results.py:255)
//   conv1       -- uint8 decode + standardise fused into block1_conv1 (3x3 s2 valid, 3->32) + BN + ReLU
//   depthwise   -- 3x3 'same' depthwise conv of every SeparableConv2D (optional ReLU on the input)
//   pool_add    -- MaxPool 3x3 s2 'same' (TF padding, -inf) + residual add
//   subsample   -- stride-2 pixel gather feeding the 1x1 s2 residual convolutions
//   gap         -- global average pooling -> 2048 features
//   head        -- Philox4x32-10 dropout masks, masked operand expansion, logits + softmax + mean/std over T
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace bq {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ void bf16x8_to_float(const uint4& v, float (&f)[8]) {
  const __nv_bfloat162* b = (const __nv_bfloat162*)&v;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 t = __bfloat1622float2(b[j]);
    f[2 * j] = t.x;
    f[2 * j + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 float_to_bf16x8(const float (&f)[8]) {
  uint4 o;
  __nv_bfloat162* b = (__nv_bfloat162*)&o;
#pragma unroll
  for (int j = 0; j < 4; ++j) b[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
  return o;
}

// ---------------------------------------------------------------------------------------------------
// per-tile statistics: exact integer sums, fp64 finish.  One block per tile.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512)
tile_stats_kernel(const uint8_t* __restrict__ tiles, int64_t bytes_per_tile, float* __restrict__ mean,
                  float* __restrict__ inv_std, const float* __restrict__ c1_sumw = nullptr,
                  const float* __restrict__ c1_scale = nullptr, const float* __restrict__ c1_shift = nullptr,
                  float* __restrict__ c1_affine = nullptr /*[n][64]: per-tile (g, h) of conv1_tc_kernel's epilogue*/,
                  float* __restrict__ c1_m0 = nullptr /*[n]: the integer the producers subtract from every pixel*/) {
  const uint8_t* src = tiles + (int64_t)blockIdx.x * bytes_per_tile;
  unsigned long long s = 0, s2 = 0;
  // head up to 16-byte alignment, vector body, tail
  const uintptr_t addr = (uintptr_t)src;
  int64_t head = (16 - (addr & 15)) & 15;
  if (head > bytes_per_tile) head = bytes_per_tile;
  const int64_t nvec = (bytes_per_tile - head) / 16;
  const uint4* vsrc = (const uint4*)(src + head);
  for (int64_t i = threadIdx.x; i < nvec; i += blockDim.x) {
    const uint4 v = __ldg(vsrc + i);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    unsigned ls = 0, ls2 = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const unsigned x = (w[k] >> (8 * b)) & 0xFFu;
        ls += x;
        ls2 += x * x;
      }
    }
    s += ls;
    s2 += ls2;
  }
  const int64_t tail0 = head + nvec * 16;
  for (int64_t i = threadIdx.x; i < head + (bytes_per_tile - tail0); i += blockDim.x) {
    const int64_t j = i < head ? i : tail0 + (i - head);
    const unsigned x = src[j];
    s += x;
    s2 += x * x;
  }
  __shared__ unsigned long long sh[2][16];
  __shared__ double stat[2];
  for (int o = 16; o; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long ts = 0, ts2 = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { ts += sh[0][w]; ts2 += sh[1][w]; }
    const double n = (double)bytes_per_tile;
    const double m = (double)ts / n;
    double var = (double)ts2 / n - m * m;
    if (var < 0.0) var = 0.0;
    double sd = sqrt(var);
    const double floor_sd = 1.0 / sqrt(n);
    if (sd < floor_sd) sd = floor_sd;
    mean[blockIdx.x] = (float)m;
    inv_std[blockIdx.x] = (float)(1.0 / sd);
    stat[0] = m; stat[1] = 1.0 / sd;
  }
  if (c1_affine) {
    // block1_conv1 is bias-free and 'valid': BN(conv(W, (x - m) / sd)) = conv(W, x - m0) * g + h with, per output channel,
    // g = scale / sd and h = shift - (m - m0) * sum(W) * g  (fp64 here, one fp32 FMA per output in the kernel).
    // m0 = round(m) is removed from the pixels BEFORE the convolution (x - m0 is an integer in [-255, 255]: still exact in
    // bf16), so the convolution never carries a large common term that the epilogue would have to cancel: on a constant
    // tile the accumulators are exactly 0, and on low-contrast tiles 1 / sd does not amplify fp32 summation rounding.
    // m and 1 / sd enter as the SAME fp32 values the standardise-first arithmetic uses (tf.image.per_image_standardization
    // and the oracle subtract an fp32 mean): on a tile where one pixel differs the fp32 mean is the constant itself.
    __syncthreads();
    const double mf = (double)(float)stat[0], isf = (double)(float)stat[1];
    const double m0 = rint(mf);
    if (threadIdx.x == 0) c1_m0[blockIdx.x] = (float)m0;
    if (threadIdx.x < 32) {
      const int c = threadIdx.x;
      const double g = isf * (double)c1_scale[c];
      c1_affine[(int64_t)blockIdx.x * 64 + c] = (float)g;
      c1_affine[(int64_t)blockIdx.x * 64 + 32 + c] = (float)((double)c1_shift[c] - (mf - m0) * (double)c1_sumw[c] * g);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// block1_conv1: uint8 NHWC [n,299,299,3] -> bf16 NHWC [n,149,149,32]; 3x3 stride 2 valid, BN, ReLU.
// A block computes a 16x16 output patch: the 33x33x3 input patch is standardised into smem as fp32 once,
// each thread owns one output pixel x 32 channels (fp32 weights broadcast from smem).
// ---------------------------------------------------------------------------------------------------
constexpr int kC1Tile = 16;
constexpr int kC1In = 2 * kC1Tile + 1;
// TIn = uint8_t: raw RGB, standardised here with the tile's (mean, 1/std).  TIn = float: the caller already applied
// tf.image.per_image_standardization (the reference's literal call, results.py:255-257) -- values are used as they are.
// A float tile holding a NaN or +-Inf would reach the output as an ordinary-looking number (fmaxf(NaN, 0) = 0), so the
// float instantiation records the smallest call-global index i0 + img of such a tile in *nonfinite (atomicMin; the
// caller resets the word to ~0 and reports it after the call).
template <typename TIn>
__global__ void __launch_bounds__(256)
conv1_kernel(const TIn* __restrict__ tiles, const float* __restrict__ mean, const float* __restrict__ inv_std,
             const float* __restrict__ w /*[27][32]*/, const float* __restrict__ scale, const float* __restrict__ shift,
             bf16* __restrict__ out, int in_px, int out_px, unsigned long long* __restrict__ nonfinite = nullptr,
             int64_t i0 = 0) {
  __shared__ float patch[kC1In * kC1In * 3];
  __shared__ __align__(16) float ws[27 * 32];
  __shared__ float sc[32], sh[32];
  const int img = blockIdx.z;
  const int oy0 = blockIdx.y * kC1Tile, ox0 = blockIdx.x * kC1Tile;
  constexpr bool kRaw = sizeof(TIn) == 1;
  const float mu = kRaw ? mean[img] : 0.f, is = kRaw ? inv_std[img] : 1.f;
  const TIn* src = tiles + (int64_t)img * in_px * in_px * 3;
  for (int i = threadIdx.x; i < 27 * 32; i += blockDim.x) ws[i] = w[i];
  if (threadIdx.x < 32) { sc[threadIdx.x] = scale[threadIdx.x]; sh[threadIdx.x] = shift[threadIdx.x]; }
  const int iy0 = oy0 * 2, ix0 = ox0 * 2;
  bool finite = true;
  for (int i = threadIdx.x; i < kC1In * kC1In * 3; i += blockDim.x) {
    const int r = i / (kC1In * 3), rem = i - r * (kC1In * 3);
    const int y = iy0 + r, xc = ix0 * 3 + rem;
    float v = 0.f;
    if (y < in_px && xc < in_px * 3) {
      const float raw = (float)src[(int64_t)y * in_px * 3 + xc];
      if constexpr (!kRaw) finite &= isfinite(raw);
      v = kRaw ? __fmul_rn(__fadd_rn(raw, -mu), is) : raw;
    }
    patch[i] = v;
  }
  // the patches of a tile's blocks cover every one of its values (the last block's reaches row / column 320 > 298)
  if constexpr (!kRaw) {
    if (!finite) atomicMin(nonfinite, (unsigned long long)(i0 + img));
  }
  __syncthreads();
  const int ty = threadIdx.x / kC1Tile, tx = threadIdx.x % kC1Tile;
  const int oy = oy0 + ty, ox = ox0 + tx;
  if (oy >= out_px || ox >= out_px) return;
  // 27 inputs x 32 channels: weights as LDS.128 broadcasts, packed fp32x2 FMAs (FFMA2) -- same per-lane RN fma
  float2 acc2[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) acc2[c] = make_float2(0.f, 0.f);
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
        const float x = patch[((2 * ty + ky) * kC1In + (2 * tx + kx)) * 3 + ci];
        const float2 xx = make_float2(x, x);
        const float4* wr = (const float4*)(ws + ((ky * 3 + kx) * 3 + ci) * 32);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 wv = wr[c4];
          acc2[2 * c4] = __ffma2_rn(xx, make_float2(wv.x, wv.y), acc2[2 * c4]);
          acc2[2 * c4 + 1] = __ffma2_rn(xx, make_float2(wv.z, wv.w), acc2[2 * c4 + 1]);
        }
      }
    }
  }
  float acc[32];
#pragma unroll
  for (int c = 0; c < 16; ++c) { acc[2 * c] = acc2[c].x; acc[2 * c + 1] = acc2[c].y; }
  bf16* o = out + (((int64_t)img * out_px + oy) * out_px + ox) * 32;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = g * 8 + j;
      f[j] = fmaxf(__fadd_rn(__fmul_rn(acc[c], sc[c]), sh[c]), 0.f);
    }
    *(uint4*)(o + g * 8) = float_to_bf16x8(f);
  }
}

// ---------------------------------------------------------------------------------------------------
// MaxPool 3x3 stride 2 'same' (TF: pad_total = max((ceil(H/2)-1)*2 + 3 - H, 0), before = total/2) + residual
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
maxpool_add_kernel(const bf16* __restrict__ in, const bf16* __restrict__ res, bf16* __restrict__ out, int n_img,
                   int H, int W, int Ho, int Wo, int C, int pad_top, int pad_left, int out_pitch = 0 /*0: dense [n, Ho, Wo, C];
                   else pixel (y, x) of image b is row b * out_pitch^2 + y * out_pitch + x (zero-padded middle-flow layout)*/) {
  const int cv = C >> 3;
  const int64_t total = (int64_t)n_img * Ho * Wo * cv;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(idx % cv);
    int64_t pix = idx / cv;
    const int xo = (int)(pix % Wo);
    pix /= Wo;
    const int yo = (int)(pix % Ho);
    const int img = (int)(pix / Ho);
    // Window taps that fall into the padding are clamped onto the nearest valid pixel: a duplicate never changes
    // a maximum, so all nine 16-byte loads are unconditional and in flight together; the max itself is exact in bf16.
    const bf16* base = in + ((int64_t)img * H * W) * C + c8 * 8;
    uint4 v[9];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int yy = min(max(yo * 2 + ky - pad_top, 0), H - 1);
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int xx = min(max(xo * 2 + kx - pad_left, 0), W - 1);
        v[ky * 3 + kx] = __ldg((const uint4*)(base + ((int64_t)yy * W + xx) * C));
      }
    }
    const uint4 rv = __ldg((const uint4*)(res + (((int64_t)img * Ho + yo) * Wo + xo) * C + c8 * 8));
    __nv_bfloat162 mx[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      __nv_bfloat162 a = ((const __nv_bfloat162*)&v[0])[q];
#pragma unroll
      for (int k = 1; k < 9; ++k) a = __hmax2(a, ((const __nv_bfloat162*)&v[k])[q]);
      mx[q] = a;
    }
    float m[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float2 f = __bfloat1622float2(mx[q]);
      m[2 * q] = f.x;
      m[2 * q + 1] = f.y;
    }
    const int64_t o = (((int64_t)img * Ho + yo) * Wo + xo) * C + c8 * 8;
    float r[8];
    bf16x8_to_float(rv, r);
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = __fadd_rn(m[j], r[j]);
    const int64_t od = out_pitch ? (((int64_t)img * out_pitch + yo) * out_pitch + xo) * C + c8 * 8 : o;
    *(uint4*)(out + od) = float_to_bf16x8(m);
  }
}

// stride-2 pixel gather: out[n,yo,xo,:] = in[n,2yo,2xo,:]   (1x1 stride-2 'valid' conv samples 0,2,4,...)
__global__ void __launch_bounds__(256)
subsample2_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, int n_img, int H, int W, int Ho, int Wo, int C,
                  int in_pitch = 0 /*0: dense input; else the zero-padded layout with this row pitch*/) {
  const int cv = C >> 3;
  const int64_t total = (int64_t)n_img * Ho * Wo * cv;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(idx % cv);
    int64_t pix = idx / cv;
    const int xo = (int)(pix % Wo);
    pix /= Wo;
    const int yo = (int)(pix % Ho);
    const int img = (int)(pix / Ho);
    const int64_t ip = in_pitch ? ((int64_t)img * in_pitch + 2 * yo) * in_pitch + 2 * xo : ((int64_t)img * H + 2 * yo) * W + 2 * xo;
    const uint4 v = __ldg((const uint4*)(in + ip * C + c8 * 8));
    *(uint4*)(out + (((int64_t)img * Ho + yo) * Wo + xo) * C + c8 * 8) = v;
  }
}

// global average pool: [n, HW, C] bf16 -> fp32 [n, C] (+ bf16 copy as the next GEMM's A operand)
__global__ void __launch_bounds__(256)
gap_kernel(const bf16* __restrict__ in, float* __restrict__ feat, bf16* __restrict__ feat_bf16, int n_img, int HW, int C) {
  const int64_t total = (int64_t)n_img * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % C);
    const int img = (int)(idx / C);
    const bf16* p = in + (int64_t)img * HW * C + c;
    float s = 0.f;
    for (int i = 0; i < HW; ++i) s += __bfloat162float(p[(int64_t)i * C]);
    const float m = s / (float)HW;
    feat[idx] = m;
    feat_bf16[idx] = __float2bfloat16_rn(m);
  }
}

// ---------------------------------------------------------------------------------------------------
// MC-dropout head pieces
// ---------------------------------------------------------------------------------------------------
struct Philox4 { uint32_t x, y, z, w; };

// Philox4x32-10 (Salmon et al. 2011); same stream as oracle/xception_uq.py:philox4x32_10
__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return {c0, c1, c2, c3};
}

// keep-bits of 4 consecutive hidden units e..e+3 of (tile, sample t, site): bit j set = keep unit e+j.
// counter = (e/4, t*4 + site, tile_lo, tile_hi), key = seed; keep iff draw >= floor(rate * 2^32).
__device__ __forceinline__ uint32_t keep4(uint64_t seed, uint64_t tile, int t, int site, int e4, uint32_t thresh) {
  const Philox4 r = philox4x32_10((uint32_t)e4, (uint32_t)(t * 4 + site), (uint32_t)tile, (uint32_t)(tile >> 32),
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
  return (r.x >= thresh ? 1u : 0u) | (r.y >= thresh ? 2u : 0u) | (r.z >= thresh ? 4u : 0u) | (r.w >= thresh ? 8u : 0u);
}

// A2[(i*T + t), k] = keep(i, t, site, k) ? h[i, k] : 0      (one thread = 4 consecutive k)
// masks (nullable): injected uint8 keep-masks [n, T, n_sites, width]; site_slot indexes dim 2.
__global__ void __launch_bounds__(256)
mc_expand_kernel(const bf16* __restrict__ h, bf16* __restrict__ a2, int n, int T, int width, uint64_t seed,
                 uint64_t tile_base, int site, uint32_t thresh, const uint8_t* __restrict__ masks, int n_sites,
                 int site_slot, int mask_w = 0) {
  if (mask_w <= 0) mask_w = width;
  const int w4 = width >> 2;
  const int64_t total = (int64_t)n * T * w4;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int e4 = (int)(idx % w4);
    const int64_t row = idx / w4;
    const int t = (int)(row % T);
    const int i = (int)(row / T);
    uint32_t kb;
    if (masks) {
      const uint8_t* mp = masks + (((int64_t)i * T + t) * n_sites + site_slot) * mask_w + e4 * 4;
      kb = (mp[0] ? 1u : 0u) | (mp[1] ? 2u : 0u) | (mp[2] ? 4u : 0u) | (mp[3] ? 8u : 0u);
    } else {
      kb = keep4(seed, tile_base + (uint64_t)i, t, site, e4, thresh);
    }
    const uint2 v = *(const uint2*)(h + (int64_t)i * width + e4 * 4);
    uint2 o;
    o.x = ((kb & 1u) ? (v.x & 0xFFFFu) : 0u) | ((kb & 2u) ? (v.x & 0xFFFF0000u) : 0u);
    o.y = ((kb & 4u) ? (v.y & 0xFFFFu) : 0u) | ((kb & 8u) ? (v.y & 0xFFFF0000u) : 0u);
    *(uint2*)(a2 + row * width + e4 * 4) = o;
  }
}

constexpr int kMaxClasses = 8;

}  // namespace bq
