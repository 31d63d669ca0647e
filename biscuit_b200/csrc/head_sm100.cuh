// Fused Monte-Carlo-dropout head (SURVEY.md K7): ONE kernel evaluates the dropout-bearing layers T times on one
// backbone feature pass and reduces to the per-tile mean prediction and dropout-sample std.
//
//   h1 [n, W]  (hidden_0 output, computed once per tile by the GEMM kernel)
//   for t in 0..T-1:   a   = keep1(tile, t) .* h1                         (Philox4x32-10, counter based, site 1)
//                      h2  = bf16( relu( (a @ W2^T) / (1-p) + b2 ) )       (tcgen05.mma, fp32 accumulation in TMEM)
//                      z   = ((keep2(tile, t) .* h2) @ W3) / (1-p) + b3    (site 2, fp32)
//                      p_t = softmax(z)
//   mean = E_t[p_t],  std = sqrt(E_t[(p_t - mean)^2])                      (population std, warp shuffles)
//
// Mapping: a work unit is 4 tiles x 32 sample slots = the 128 rows of one UMMA M tile, arranged so that TMEM lane
// quadrant q (= epilogue warp q) holds exactly the samples of tile q.  The masked A operand is never materialised in
// HBM: the four "row" warps generate each 128x64 k-block straight into the 128B-swizzled smem stage (16 Philox
// draws + eight 16-byte selects per thread), W2 k-blocks arrive by TMA, and the 128 x 512 fp32 accumulator of one
// output half fills the whole TMEM (512 columns).  The epilogue reads it back with tcgen05.ld, applies bias / ReLU /
// bf16 rounding / the second mask and folds the 1024->C prelogits layer into per-row partial logits, so h2 never
// leaves the SM either.  T > 32 is handled by looping sample chunks and merging (n, mean, M2) with Chan's formula.
#pragma once

#include "gemm_sm100.cuh"
#include "layers.cuh"

namespace bq {
namespace head {

using namespace sm100;

constexpr int kHStages = 2;
constexpr int kHABytes = 128 * 64 * 2;            // 16 KB: masked activations, one k-block
constexpr int kHBBytes = 512 * 64 * 2;            // 64 KB: W2 rows of one output half, one k-block (2 TMA boxes)
constexpr int kHStageBytes = kHABytes + kHBBytes;
constexpr int kHMaxW = 1024;
constexpr int kHThreads = 192;                    // warp 0: TMA (W2), warp 1: TMEM + MMA issue, warps 2-5: rows

struct HeadParams {
  const bf16* h1;           // [n, W] bf16
  const float* b2;          // [W]
  const float* w3;          // [W][C] fp32
  const float* b3;          // [C]
  float* mean;              // [n, C]
  float* stdv;              // [n, C]
  const uint8_t* masks;     // nullable injected keep-masks [n, T, n_sites, mask_w]
  int n, T, W, C;
  int n_sites, slot1, slot2; // enabled sites in the mask tensor; slot < 0: that site has no dropout (keep everything)
  int mask_w;               // row pitch of the injected masks (2048 when the feature site is enabled, else W)
  int w2_box;               // rows of one W2 TMA box: 256, or W itself when W < 256 (bn_box_for in model.cu)
  int h1_per_sample;        // 1: h1 is [n * T, W] (dropout on the pooled features made hidden_0 sample dependent)
  float inv_keep1, inv_keep2;   // 1/(1-p) behind an enabled site, 1 otherwise
  float inv_keep;
  uint32_t thresh;
  uint64_t seed, tile_base;
};

struct HeadSmem {
  static constexpr int kStageOff = 0;
  static constexpr int kH1Off = kHStages * kHStageBytes;                 // bf16 [4][kHMaxW]
  static constexpr int kB2Off = kH1Off + 4 * kHMaxW * 2;                 // float [kHMaxW]
  static constexpr int kW3Off = kB2Off + kHMaxW * 4;                     // float [kHMaxW][2..8] (C <= 8)
  static constexpr int kBarOff = kW3Off + kHMaxW * kMaxClasses * 4;
  static constexpr int kTotal = kBarOff + 256 + 1024;
};

__device__ __forceinline__ uint32_t keep8(const HeadParams& p, uint64_t tile, int tile_local, int t, int site, int slot,
                                          int k) {
  if (slot < 0) return 0xFFu;                       // no dropout at this site
  if (p.masks) {
    const uint8_t* mp = p.masks + (((int64_t)tile_local * p.T + t) * p.n_sites + slot) * p.mask_w + k;
    const uint2 m = *(const uint2*)mp;
    uint32_t kb = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      kb |= ((m.x >> (8 * j)) & 0xFFu) ? (1u << j) : 0u;
      kb |= ((m.y >> (8 * j)) & 0xFFu) ? (1u << (4 + j)) : 0u;
    }
    return kb;
  }
  return keep4(p.seed, tile, t, site, k >> 2, p.thresh) | (keep4(p.seed, tile, t, site, (k >> 2) + 1, p.thresh) << 4);
}

__global__ void __launch_bounds__(kHThreads, 1)
mc_head_fused_kernel(const __grid_constant__ CUtensorMap tmap_w2 /*[W(out), W(in)] bf16, box [w2_box x 64]*/,
                     const HeadParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + HeadSmem::kBarOff;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kHStages + s); };
  const uint32_t acc_full = bar_base + 8u * (2 * kHStages);
  const uint32_t acc_empty = bar_base + 8u * (2 * kHStages + 1);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kHStages + 2);
  volatile uint32_t* tmem_slot_ptr = (volatile uint32_t*)(smem_gen + HeadSmem::kBarOff + 8 * (2 * kHStages + 2));
  bf16* s_h1 = (bf16*)(smem_gen + HeadSmem::kH1Off);
  float* s_b2 = (float*)(smem_gen + HeadSmem::kB2Off);
  float* s_w3 = (float*)(smem_gen + HeadSmem::kW3Off);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int W = p.W, C = p.C;
  const int num_kb = W / 64;
  const int n_halves = (W + 511) / 512;
  const int n_groups = (p.n + 3) / 4;
  const int n_chunks = (p.T + 31) / 32;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_w2);
    for (int s = 0; s < kHStages; ++s) { mbar_init(full_bar(s), 5); mbar_init(empty_bar(s), 1); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = threadIdx.x; i < W; i += blockDim.x) s_b2[i] = __ldg(p.b2 + i);
  for (int i = threadIdx.x; i < W * C; i += blockDim.x) s_w3[i] = __ldg(p.w3 + i);
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  // every role walks the same (group, chunk, half, k-block) sequence
  int s = 0; uint32_t ph = 0;        // smem ring
  uint32_t acc_ph = 0;               // accumulator full/empty phase

  for (int g = blockIdx.x; g < n_groups; g += gridDim.x) {
    // stage the four tiles' hidden_0 activations (all threads), visible to the row warps after the barrier
    __syncthreads();
    for (int i = threadIdx.x; i < 4 * W / 8; i += blockDim.x) {
      const int tl = i / (W / 8), v = i % (W / 8);
      const int tile = g * 4 + tl;
      uint4 val = make_uint4(0u, 0u, 0u, 0u);
      if (tile < p.n && !p.h1_per_sample) val = __ldg((const uint4*)(p.h1 + (int64_t)tile * W + v * 8));
      *(uint4*)(s_h1 + tl * kHMaxW + v * 8) = val;
    }
    __syncthreads();

    // per-tile running statistics over sample chunks (row warps only use them)
    float r_n = 0.f, r_mean[kMaxClasses], r_m2[kMaxClasses];
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) { r_mean[c] = 0.f; r_m2[c] = 0.f; }

    for (int sc = 0; sc < n_chunks; ++sc) {
      float logit[kMaxClasses];
#pragma unroll
      for (int c = 0; c < kMaxClasses; ++c) logit[c] = 0.f;
      for (int h = 0; h < n_halves; ++h) {
        const int hw = min(512, W - h * 512);                  // output units of this half
        if (warp == 0) {
          // ---------------- W2 k-blocks by TMA ----------------
          // A box is 256 rows, or all W rows when W < 256 (then one box covers the half): either way box nb lands at
          // row nb * 256 of the stage, where the MMA below reads it.  Rows past W arrive zero-filled and count in full.
          if (lane == 0) {
            const int box = p.w2_box;
            for (int kb = 0; kb < num_kb; ++kb) {
              mbar_wait(empty_bar(s), ph ^ 1u);
              mbar_expect_tx(full_bar(s), (uint32_t)((hw + box - 1) / box) * (uint32_t)box * 64u * 2u);
              const uint32_t b_dst = smem_base + s * kHStageBytes + kHABytes;
              for (int nb = 0; nb * box < hw; ++nb)
                tma_load_2d(b_dst + nb * box * 128, &tmap_w2, full_bar(s), kb * 64, h * 512 + nb * box);
              if (++s == kHStages) { s = 0; ph ^= 1u; }
            }
          }
        } else if (warp == 1) {
          // ---------------- MMA issue ----------------
          if (lane == 0) {
            mbar_wait(acc_empty, acc_ph ^ 1u);
            tc_fence_after();
            for (int kb = 0; kb < num_kb; ++kb) {
              mbar_wait(full_bar(s), ph);
              tc_fence_after();
              const uint32_t a_src = smem_base + s * kHStageBytes, b_src = a_src + kHABytes;
              const uint64_t da = make_smem_desc<128>(a_src);
              for (int nb = 0; nb * 256 < hw; ++nb) {
                const int ncols = min(256, hw - nb * 256);
                const uint32_t idesc = make_idesc(128, ncols);
                const uint64_t db = make_smem_desc<128>(b_src + nb * 256 * 128);
                for (int k = 0; k < 4; ++k)
                  umma_bf16(tmem_base + (uint32_t)(nb * 256), da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc,
                            (kb | k) ? 1u : 0u);
              }
              umma_commit(empty_bar(s));
              if (kb == num_kb - 1) umma_commit(acc_full);
              if (++s == kHStages) { s = 0; ph ^= 1u; }
            }
          }
        } else {
          // ---------------- row warps: masked A operand, then the epilogue of this half ----------------
          const int q = warp & 3;                               // TMEM lane quadrant == tile slot of this warp
          const int row = q * 32 + lane;
          const int tile_local = g * 4 + q;
          const int t = sc * 32 + lane;
          const bool valid = tile_local < p.n && t < p.T;
          const uint64_t tile = p.tile_base + (uint64_t)tile_local;
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(empty_bar(s), ph ^ 1u);
            uint8_t* a_dst = smem_gen + s * kHStageBytes + (size_t)row * 128;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int k = kb * 64 + j * 8;
              uint4 v;
              if (p.h1_per_sample) {                                      // one hidden_0 row per (tile, sample)
                v = valid ? __ldg((const uint4*)(p.h1 + ((int64_t)tile_local * p.T + t) * W + k)) : make_uint4(0u, 0u, 0u, 0u);
              } else {
                v = *(const uint4*)(s_h1 + q * kHMaxW + k);              // broadcast within the warp
              }
              const uint32_t kb8 = valid ? keep8(p, tile, tile_local, t, 1, p.slot1, k) : 0u;
              v.x = ((kb8 & 1u) ? (v.x & 0xFFFFu) : 0u) | ((kb8 & 2u) ? (v.x & 0xFFFF0000u) : 0u);
              v.y = ((kb8 & 4u) ? (v.y & 0xFFFFu) : 0u) | ((kb8 & 8u) ? (v.y & 0xFFFF0000u) : 0u);
              v.z = ((kb8 & 16u) ? (v.z & 0xFFFFu) : 0u) | ((kb8 & 32u) ? (v.z & 0xFFFF0000u) : 0u);
              v.w = ((kb8 & 64u) ? (v.w & 0xFFFFu) : 0u) | ((kb8 & 128u) ? (v.w & 0xFFFF0000u) : 0u);
              *(uint4*)(a_dst + ((j ^ (row & 7)) << 4)) = v;
            }
            fence_async_smem();                                 // generic writes -> visible to the tensor core (async proxy)
            __syncwarp();
            if (lane == 0) mbar_arrive(full_bar(s));
            if (++s == kHStages) { s = 0; ph ^= 1u; }
          }
          // epilogue of this half: bias, ReLU, bf16 rounding, second mask, prelogits partial sums
          mbar_wait(acc_full, acc_ph);
          tc_fence_after();
          const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16);
          for (int c0 = 0; c0 < hw; c0 += 32) {
            uint32_t v[32];
            tmem_ld_32x32b_x32(t_row + (uint32_t)c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              const int n0 = h * 512 + c0 + j8 * 8;
              const uint32_t kb8 = valid ? keep8(p, tile, tile_local, t, 2, p.slot2, n0) : 0u;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                float x = __fadd_rn(__fmul_rn(__uint_as_float(v[j8 * 8 + j]), p.inv_keep1), s_b2[n0 + j]);
                x = __bfloat162float(__float2bfloat16_rn(fmaxf(x, 0.f)));      // h2 is a bf16 activation
                x = (kb8 >> j) & 1u ? x : 0.f;
#pragma unroll
                for (int c = 0; c < kMaxClasses; ++c)
                  if (c < C) logit[c] = fmaf(x, s_w3[(n0 + j) * C + c], logit[c]);
              }
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(acc_empty);
        }
        acc_ph ^= 1u;
      }  // halves

      if (warp >= 2) {
        // softmax of this sample, then warp-shuffle statistics over the <= 32 samples of the chunk
        const int q = warp & 3;
        const int tile_local = g * 4 + q;
        const int t = sc * 32 + lane;
        const bool valid = tile_local < p.n && t < p.T;
        float z[kMaxClasses], mx = -INFINITY, den = 0.f;
#pragma unroll
        for (int c = 0; c < kMaxClasses; ++c)
          if (c < C) { z[c] = __fadd_rn(__fmul_rn(logit[c], p.inv_keep2), __ldg(p.b3 + c)); mx = fmaxf(mx, z[c]); }
#pragma unroll
        for (int c = 0; c < kMaxClasses; ++c)
          if (c < C) { z[c] = expf(z[c] - mx); den += z[c]; }
        const unsigned vm = __ballot_sync(0xffffffffu, valid);
        const float cn = (float)__popc(vm);
        if (cn > 0.f) {
#pragma unroll
          for (int c = 0; c < kMaxClasses; ++c) {
            if (c >= C) continue;
            const float pr = valid ? z[c] / den : 0.f;
            float sum = pr;
            for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            const float cm = sum / cn;
            const float d = valid ? pr - cm : 0.f;
            float m2 = d * d;
            for (int o = 16; o; o >>= 1) m2 += __shfl_xor_sync(0xffffffffu, m2, o);
            if (r_n == 0.f) {                       // first (for T <= 32: only) chunk: plain two-pass mean / M2
              r_mean[c] = cm;
              r_m2[c] = m2;
            } else {                                // Chan et al. merge of (r_n, r_mean, r_m2) with (cn, cm, m2)
              const float tot = r_n + cn, delta = cm - r_mean[c];
              r_mean[c] += delta * cn / tot;
              r_m2[c] += m2 + delta * delta * r_n * cn / tot;
            }
          }
          r_n += cn;
        }
      }
    }  // sample chunks

    if (warp >= 2 && lane == 0) {
      const int tile_local = g * 4 + (warp & 3);
      if (tile_local < p.n) {
#pragma unroll
        for (int c = 0; c < kMaxClasses; ++c) {
          if (c >= C) continue;
          p.mean[(int64_t)tile_local * C + c] = r_mean[c];
          p.stdv[(int64_t)tile_local * C + c] = sqrtf(r_m2[c] / r_n);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace head
}  // namespace bq
