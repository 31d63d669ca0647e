// Xception-UQ Monte-Carlo-dropout inference: weight packing, static execution plan, C ABI.
//
// Replaces slideflow.model.tensorflow.UncertaintyInterface.__call__ (call site: reference results.py:234,257;
// architecture contract: reference biscuit/hp.py:3-24).  One backbone pass per tile, T dropout-head samples on
// the pooled features (the reference schedule repeats the whole network T times; the backbone is deterministic in
// inference mode, so the results are identical).  Layer list / padding rules: SURVEY.md Appendix B, restated in
// oracle/xception_uq.py which is the parity checker for this file.
#include <cuda.h>

#include <cmath>
#include <cstdlib>
#include <map>
#include <memory>

#include "encoded.cuh"
#include "gemm_sm100.cuh"
#include "layers.cuh"
#include "head_sm100.cuh"
#include "dwpipe_sm100.cuh"
#include "sepconv2d_sm100.cuh"
#include "sepmid_sm100.cuh"
#include "conv1_sm100.cuh"
#include "stain_sm100.cuh"

int bq_stain_launch(bq_ctx* ctx, const uint8_t* tiles_dev, int64_t n, int32_t px, const float* lut_dev, float* stats_dev,
                    const float target_means[3], const float target_stds[3], uint8_t* out_dev);   // stain.cu

using bq::bf16;
using bq::GemmParams;

namespace {

constexpr float kBnEps = 1e-3f;
constexpr int kFeatures = 2048;

// ------------------------------------------------------------------------------------------------
// TMA descriptors (driver entry point fetched at run time: the library links only the static cudart)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2-D bf16 K-major matrix [rows, cols] with row pitch `ld` elements; box = [box_rows, box_cols]
int make_tmap(bq_ctx* ctx, CUtensorMap* out, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld,
              uint32_t box_rows, uint32_t box_cols, bool no_swizzle = false) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return bq_fail(ctx, BQ_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * sizeof(bf16)};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapSwizzle swz = no_swizzle ? CU_TENSOR_MAP_SWIZZLE_NONE
                           : box_cols * sizeof(bf16) == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                           : box_cols * sizeof(bf16) == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                           : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return bq_fail(ctx, BQ_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu box=%ux%u", (int)r,
                   (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_cols);
  return BQ_OK;
}

// 4-D NHWC bf16 activation [N, H, W, C] with a [1, box_h, box_w, box_c] box, no swizzle (depthwise halo tiles)
int make_tmap_nhwc(bq_ctx* ctx, CUtensorMap* out, const void* ptr, uint64_t n, uint64_t h, uint64_t w, uint64_t c,
                   uint32_t box_h, uint32_t box_w, uint32_t box_c, bool swizzle128 = false, bool swizzle64 = false,
                   uint64_t pitch = 0 /*rows and columns of the (zero-padded) storage, 0 = dense*/) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return bq_fail(ctx, BQ_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[4] = {c, w, h, n};
  const uint64_t pw = pitch ? pitch : w, ph = pitch ? pitch : h;
  cuuint64_t strides[3] = {c * sizeof(bf16), pw * c * sizeof(bf16), ph * pw * c * sizeof(bf16)};
  cuuint32_t box[4] = {box_c, box_w, box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : (swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE),
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return bq_fail(ctx, BQ_ERR_CUDA, "cuTensorMapEncodeTiled(4d) failed (%d)", (int)r);
  return BQ_OK;
}

// ------------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------------
struct PwWeights {          // a GEMM's B operand + per-channel epilogue
  int cin = 0, cout = 0, ktot = 0;
  DevBuf w;                 // bf16 [cout][ktot]
  DevBuf scale, shift;      // fp32 [cout]
};
struct SepWeights {
  DevBuf dw;                // fp32 [9][cin]
  PwWeights pw;
};

struct TensorIndex {
  std::map<std::string, const bq_named_tensor*> by_name;
  const bq_named_tensor* find(const std::string& n) const {
    auto it = by_name.find(n);
    return it == by_name.end() ? nullptr : it->second;
  }
};

inline uint16_t f32_to_bf16_rne(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((u >> 16) | 0x40);   // NaN
  u += 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

int upload(bq_ctx* ctx, DevBuf& dst, const void* src, size_t bytes) {
  int rc = bq_alloc(ctx, dst, bytes);
  if (rc) return rc;
  BQ_CUDA(ctx, cudaMemcpy(dst.p, src, bytes, cudaMemcpyHostToDevice));
  return BQ_OK;
}

int need(bq_ctx* ctx, const TensorIndex& ti, const std::string& name, std::initializer_list<int64_t> shape,
         const bq_named_tensor** out) {
  const bq_named_tensor* t = ti.find(name);
  if (!t) return bq_fail(ctx, BQ_ERR_WEIGHTS, "missing weight tensor '%s'", name.c_str());
  if (t->ndim != (int)shape.size()) return bq_fail(ctx, BQ_ERR_WEIGHTS, "'%s': expected %d dims, got %d", name.c_str(), (int)shape.size(), t->ndim);
  int i = 0;
  for (int64_t s : shape) {
    if (t->shape[i] != s) return bq_fail(ctx, BQ_ERR_WEIGHTS, "'%s': dim %d is %lld, expected %lld", name.c_str(), i, (long long)t->shape[i], (long long)s);
    ++i;
  }
  if (!t->data) return bq_fail(ctx, BQ_ERR_WEIGHTS, "'%s': null data", name.c_str());
  *out = t;
  return BQ_OK;
}

// BatchNorm (inference) -> y = x*scale + shift, eps = 1e-3 (Keras Xception)
int load_bn(bq_ctx* ctx, const TensorIndex& ti, const std::string& bn, int c, PwWeights& w) {
  const bq_named_tensor *g, *b, *m, *v;
  int rc;
  if ((rc = need(ctx, ti, bn + "/gamma", {c}, &g)) || (rc = need(ctx, ti, bn + "/beta", {c}, &b)) ||
      (rc = need(ctx, ti, bn + "/moving_mean", {c}, &m)) || (rc = need(ctx, ti, bn + "/moving_variance", {c}, &v)))
    return rc;
  std::vector<float> sc(c), sh(c);
  for (int i = 0; i < c; ++i) {
    volatile float s = g->data[i] / sqrtf(v->data[i] + kBnEps);
    volatile float ms = m->data[i] * s;
    sc[i] = s;
    sh[i] = b->data[i] - ms;
  }
  if ((rc = upload(ctx, w.scale, sc.data(), c * 4)) || (rc = upload(ctx, w.shift, sh.data(), c * 4))) return rc;
  return BQ_OK;
}

// Keras kernel [kh,kw,cin,cout] (HWIO) -> bf16 [cout][kh*kw*cin]  (tap-major K, K-major rows)
int load_conv_gemm(bq_ctx* ctx, const TensorIndex& ti, const std::string& name, const std::string& var, int kh,
                   int cin, int cout, PwWeights& w) {
  const bq_named_tensor* k;
  int rc = need(ctx, ti, name + "/" + var, {kh, kh, cin, cout}, &k);
  if (rc) return rc;
  const int ktot = kh * kh * cin;
  std::vector<uint16_t> h((size_t)cout * ktot);
  for (int t = 0; t < kh * kh; ++t)
    for (int c = 0; c < cin; ++c)
      for (int o = 0; o < cout; ++o)
        h[(size_t)o * ktot + t * cin + c] = f32_to_bf16_rne(k->data[((size_t)t * cin + c) * cout + o]);
  w.cin = cin; w.cout = cout; w.ktot = ktot;
  if ((rc = upload(ctx, w.w, h.data(), h.size() * 2))) return rc;
  return load_bn(ctx, ti, name + "_bn", cout, w);
}

int load_dense(bq_ctx* ctx, const TensorIndex& ti, const std::string& name, int cin, int cout, PwWeights& w) {
  const bq_named_tensor *k, *b;
  int rc;
  if ((rc = need(ctx, ti, name + "/kernel", {cin, cout}, &k)) || (rc = need(ctx, ti, name + "/bias", {cout}, &b))) return rc;
  std::vector<uint16_t> h((size_t)cout * cin);
  for (int c = 0; c < cin; ++c)
    for (int o = 0; o < cout; ++o) h[(size_t)o * cin + c] = f32_to_bf16_rne(k->data[(size_t)c * cout + o]);
  w.cin = cin; w.cout = cout; w.ktot = cin;
  if ((rc = upload(ctx, w.w, h.data(), h.size() * 2))) return rc;
  return upload(ctx, w.shift, b->data, cout * 4);   // scale stays null -> alpha
}

// ------------------------------------------------------------------------------------------------
// execution plan
// ------------------------------------------------------------------------------------------------
enum OpKind { OP_STATS, OP_CONV1, OP_GEMM, OP_DW, OP_POOLADD, OP_SUBSAMPLE, OP_GAP, OP_SEP2D, OP_SEPMID };

struct Op {
  OpKind kind;
  int stage = 0;              // profiling bucket
  std::string tag;            // non-empty: a named stage output (debug hook)
  // generic tensor geometry (per tile)
  const bf16* in = nullptr;
  const bf16* in2 = nullptr;
  bf16* out = nullptr;
  int H = 0, W = 0, C = 0, Ho = 0, Wo = 0, Cout = 0;
  int relu_in = 0, pad_top = 0, pad_left = 0;
  const float* dw = nullptr;
  bq::sep2d::Sep2dParams s2;  // OP_SEP2D
  bq::sepmid::SepMidParams sm; // OP_SEPMID
  bool padded_out = false;    // the op's output is in the zero-padded 20 x 20 layout (debug-stage copies strip it)
  int in_pitch = 0, out_pitch = 0;   // OP_SUBSAMPLE input / OP_POOLADD output in the zero-padded layout (row pitch), 0 = dense
  // gemm
  GemmParams gp;
  int rows_per_tile = 0;      // M = rows_per_tile * batch
  int blk_k = 64;
  CUtensorMap ta, tb, tc, tr; // A, B, output, residual
  CUtensorMap tb2;            // B with a half-height box (2-CTA kernel: each CTA stages N/2 rows)
};

struct Arena {                // activation scratch: a handful of max-size buffers
  DevBuf buf[5];
  bf16* p(int i) { return (bf16*)buf[i].p; }
};

}  // namespace

struct bq_model {
  bq_ctx* ctx = nullptr;
  bq_model_config cfg{};
  bool weights_loaded = false;
  bool use_simt = false;                       // BQ_GEMM=simt: plain CUDA-core GEMM instead of tcgen05 (debug oracle, never the default)
  // The launch sequence of a full micro-batch after block1_conv1 is static (fixed arena addresses, tensor maps by
  // value): it is captured once into a CUDA graph and replayed, which removes ~90 stream launches per micro-batch
  // from the host and shortens the gaps between dependent kernels (BQ_GRAPH=off: plain stream launches).
  bool use_graph = true;
  cudaGraphExec_t backbone_graph = nullptr;
  int64_t graph_kernels = 0;                   // kernel launches one replay stands for (bq_launch_count bookkeeping)
  bool sep_mid = true;                         // fused depthwise->pointwise kernel on the zero-padded layout for the 728-wide middle flow (BQ_SEPMID=off)
  DevBuf midbuf[4];                            // dedicated zero-bordered [max_batch * 400 (+ slack), 728] activation buffers of the middle flow
  int max_batch = 0;
  int px = 299;

  // weights
  DevBuf conv1_w, conv1_scale, conv1_shift;    // fp32 [27][32], [32], [32]
  DevBuf conv1_wtc, conv1_sumw;                // tensor-core form of the same filter: bf16 [96][32] (hi | mid | lo thirds of fp32), fp32 [32] tap sums
  DevBuf conv1_affine, conv1_m0;               // fp32 [max_batch][64] + [max_batch]: per-tile constants of conv1_tc_kernel (tile_stats_kernel)
  PwWeights conv2;
  std::map<std::string, std::unique_ptr<SepWeights>> sep;
  std::map<std::string, std::unique_ptr<PwWeights>> res;
  std::vector<std::unique_ptr<PwWeights>> hidden;
  DevBuf w3, b3;                               // fp32 [width][classes], [classes]

  // buffers
  DevBuf tiles_dev;                            // uint8 staging [max_batch, px, px, 3] (double-buffered with tiles_dev2)
  DevBuf tiles_dev2;
  DevBuf tiles_f32[2];                         // float32 staging for already-standardised host tiles (allocated on first use)
  bool input_f32 = false;                      // the current call feeds standardised float tiles: no statistics, no normaliser
  int norm_kind = 0;                           // BQ_NORM_*: stain normalisation in front of the tile statistics
  float norm_means[3] = {0, 0, 0}, norm_stds[3] = {1, 1, 1};
  DevBuf tiles_norm, norm_lut, norm_stats;     // normalised micro-batch, gamma table, per-tile LAB statistics
  const uint8_t* tiles_src = nullptr;          // where stats / conv1 read the current micro-batch from
  cudaStream_t copy_stream = nullptr;          // H2D of micro-batch i+1 overlaps the backbone of micro-batch i
  cudaEvent_t copied[2] = {}, consumed[2] = {};
  bq_encoded* jpeg = nullptr;                  // bq_predict_uq_jpeg: descriptors, compressed staging and decode scratch
  bq_encoded* png = nullptr;                   // bq_predict_uq_png: likewise
  DevBuf mean, inv_std;                        // fp32 [max_batch]
  Arena arena;
  DevBuf feat, feat_bf16;                      // [max_batch, 2048]
  DevBuf h_act[2];                             // head activations: [max_batch * T, width] bf16 (ping-pong)
  DevBuf a2;                                   // masked operand [max_batch * T, width]
  DevBuf a0;                                   // feature-site masked operand [max_batch * T, 2048] (dropout site 0 only)
  int sites = 6;                               // dropout-site bitmask (bq_model_config.dropout_sites)
  int n_sites = 2, slot[3] = {-1, 0, 1};       // enabled sites and each site's slot in an injected mask tensor
  int mask_w = 0;                              // row pitch of injected masks
  DevBuf out_mean, out_std;                    // [max_batch, classes]
  DevBuf masks_dev;
  int head_T_cap = 0;

  std::vector<Op> plan;
  // head GEMM descriptors are rebuilt when T changes
  struct HeadGemm { GemmParams gp; CUtensorMap ta, tb, tc, tb2; };
  std::vector<HeadGemm> head_gemms;
  int head_T = -1;
  int head_batch = 0;                          // tiles accumulated before one fused-head launch (>= max_batch)

  int profiling = 0;                           // 0 off, 1 per stage, 2 per kernel family
  cudaEvent_t ev[9] = {};
  float stage_ms[8] = {};
  // per-kernel-family accounting (profiling == 2): event pair around every launch
  std::vector<cudaEvent_t> kev;
  struct KRec { int kind; double flops, bytes; };
  std::vector<KRec> krec;
  double k_ms[BQ_PROFILE_KINDS] = {}, k_flops[BQ_PROFILE_KINDS] = {}, k_bytes[BQ_PROFILE_KINDS] = {};
  int64_t k_launches[BQ_PROFILE_KINDS] = {};
};

namespace {

int same_pad_before(int h) {   // TF 'SAME', k=3, s=2
  const int out = (h + 1) / 2;
  int total = (out - 1) * 2 + 3 - h;
  if (total < 0) total = 0;
  return total / 2;
}

// profiling == 2: event pair around one launch, tagged with its kernel family and algorithmic work
struct KScope {
  bq_model* m; bool on;
  KScope(bq_model* m_, int kind, double flops, double bytes) : m(m_), on(m_->profiling == 2) {
    if (!on) return;
    const size_t i = m->krec.size();
    while (m->kev.size() < 2 * (i + 1)) { cudaEvent_t e; cudaEventCreate(&e); m->kev.push_back(e); }
    m->krec.push_back({kind, flops, bytes});
    cudaEventRecord(m->kev[2 * i], m->ctx->stream);
  }
  ~KScope() { if (on) cudaEventRecord(m->kev[2 * (m->krec.size() - 1) + 1], m->ctx->stream); }
};

void kprofile_collect(bq_model* m) {
  if (m->profiling != 2) return;
  cudaStreamSynchronize(m->ctx->stream);
  for (size_t i = 0; i < m->krec.size(); ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, m->kev[2 * i], m->kev[2 * i + 1]) != cudaSuccess) continue;
    const int k = m->krec[i].kind;
    m->k_ms[k] += ms; m->k_flops[k] += m->krec[i].flops; m->k_bytes[k] += m->krec[i].bytes; m->k_launches[k]++;
  }
  m->krec.clear();
}

int launch_gemm(bq_model* m, const GemmParams& gp, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
                const CUtensorMap& tr, int blk_k, const CUtensorMap* tb_half = nullptr) {
  bq_ctx* ctx = m->ctx;
  if (gp.M <= 0) return BQ_OK;
  if (m->use_simt) {
    dim3 grid((gp.N + 31) / 32, (gp.M + 31) / 32), block(32, 32);
    bq::gemm_simt_kernel<<<grid, block, 0, ctx->stream>>>(gp);
    BQ_LAUNCH_CHECK(ctx);
    return BQ_OK;
  }
  using namespace bq::sm100;
  const int m_tiles = (gp.M + kBM - 1) / kBM;
  const int n_tiles = (gp.N + gp.bn_box - 1) / gp.bn_box;
  if (blk_k == 32) {
    // block1_conv2: input-stationary implicit GEMM
    if (!(gp.conv_mode && gp.N == 64 && gp.K == 288 && 2 * gp.in_w + 2 + 128 <= kC2WinRows))
      return bq_fail(ctx, BQ_ERR_ARG, "conv3x3_is_kernel: unsupported geometry");
    const int g2 = m_tiles < ctx->num_sms ? m_tiles : ctx->num_sms;
    conv3x3_is_kernel<<<g2, kC2Threads, kC2Smem, ctx->stream>>>(ta, tb, tc, gp);
  } else {
    if (!tb_half || gp.bn_box % 32 != 0 || gp.N > k2MaxN)
      return bq_fail(ctx, BQ_ERR_ARG, "gemm_tcgen05_2cta_kernel: unsupported N = %d (tile %d)", gp.N, gp.bn_box);
    const int pair_tiles = ((gp.M + 2 * kBM - 1) / (2 * kBM)) * n_tiles;
    const int clusters = pair_tiles < ctx->num_sms / 2 ? pair_tiles : ctx->num_sms / 2;
    // a deeper operand ring where no residual staging is needed (the ring is what hides the DRAM round trip of A)
    if (gp.residual)
      gemm_tcgen05_2cta_kernel<k2Stages><<<2 * clusters, k2Threads, SmemPlan2<k2Stages>::kTotal, ctx->stream>>>(ta, *tb_half, tc, tr, gp);
    else
      gemm_tcgen05_2cta_kernel<k2Stages + 1><<<2 * clusters, k2Threads, SmemPlan2<k2Stages + 1>::kTotalNoRes, ctx->stream>>>(ta, *tb_half, tc, tr, gp);
  }
  BQ_LAUNCH_CHECK(ctx);
  return BQ_OK;
}

int bn_box_for(int n) {
  int r = (n + 15) & ~15;
  return r > 256 ? 256 : r;
}

// build a pointwise / dense GEMM op: A = [rows, K] activations at `a`, B = w, out = [rows, N]
int make_gemm(bq_model* m, Op& op, const bf16* a, int rows_per_tile, const PwWeights& w, bf16* out, int relu,
              const bf16* residual, float alpha = 1.0f) {
  op.kind = OP_GEMM;
  op.rows_per_tile = rows_per_tile;
  op.blk_k = 64;
  GemmParams& g = op.gp;
  g = GemmParams();
  g.M = rows_per_tile * m->max_batch;
  g.N = w.cout;
  g.K = w.ktot;
  g.bn_box = bn_box_for(w.cout);
  g.scale = (const float*)w.scale.p;
  g.shift = (const float*)w.shift.p;
  g.alpha = alpha;
  g.residual = residual;
  g.ldr = w.cout;
  g.out = out;
  g.ldc = w.cout;
  g.relu = relu;
  g.a_ptr = a; g.lda = w.ktot; g.a_rows = (long long)g.M;
  g.b_ptr = (const bf16*)w.w.p; g.ldb = w.ktot;
  int rc;
  if ((rc = make_tmap(m->ctx, &op.ta, a, (uint64_t)g.M, (uint64_t)w.ktot, (uint64_t)w.ktot, 128, 64))) return rc;
  if ((rc = make_tmap(m->ctx, &op.tb, w.w.p, (uint64_t)w.cout, (uint64_t)w.ktot, (uint64_t)w.ktot, g.bn_box, 64))) return rc;
  if ((rc = make_tmap(m->ctx, &op.tc, out, (uint64_t)g.M, (uint64_t)w.cout, (uint64_t)w.cout, 128, 64))) return rc;
  op.tr = op.tc;
  if (residual && (rc = make_tmap(m->ctx, &op.tr, residual, (uint64_t)g.M, (uint64_t)w.cout, (uint64_t)w.cout, 128, 64))) return rc;
  if ((rc = make_tmap(m->ctx, &op.tb2, w.w.p, (uint64_t)w.cout, (uint64_t)w.ktot, (uint64_t)w.ktot, g.bn_box / 2, 64))) return rc;
  return BQ_OK;
}

int build_plan(bq_model* m) {
  bq_ctx* ctx = m->ctx;
  const int B = m->max_batch;
  // the fused head is launched once per `head_batch` tiles so that it has >= 148 four-tile groups to spread over the SMs
  m->head_batch = ((592 + B - 1) / B) * B;
  if (m->head_batch < B) m->head_batch = B;
  const int px = m->px;
  const int s1 = (px - 3) / 2 + 1;        // 149
  const int s2 = s1 - 2;                  // 147
  // arena: every buffer can hold the largest activation of the net: [B, s2, s2, 128]
  const size_t max_elems = (size_t)B * s2 * s2 * 128;
  for (auto& b : m->arena.buf) {
    int rc = bq_alloc(ctx, b, max_elems * sizeof(bf16) + 1024);
    if (rc) return rc;
    BQ_CUDA(ctx, cudaMemset(b.p, 0, max_elems * sizeof(bf16) + 1024));
  }
  int rc;
  if ((rc = bq_alloc(ctx, m->tiles_dev, (size_t)B * px * px * 3 + 64)) ||
      (rc = bq_alloc(ctx, m->tiles_dev2, (size_t)B * px * px * 3 + 64)) || (rc = bq_alloc(ctx, m->mean, B * 4)) ||
      (rc = bq_alloc(ctx, m->inv_std, B * 4)) || (rc = bq_alloc(ctx, m->conv1_affine, (size_t)B * 64 * 4)) || (rc = bq_alloc(ctx, m->conv1_m0, (size_t)B * 4)) || (rc = bq_alloc(ctx, m->feat, (size_t)B * kFeatures * 4)) ||
      (rc = bq_alloc(ctx, m->feat_bf16, (size_t)B * kFeatures * 2)) ||
      (rc = bq_alloc(ctx, m->out_mean, (size_t)m->head_batch * m->cfg.n_classes * 4)) ||
      (rc = bq_alloc(ctx, m->out_std, (size_t)m->head_batch * m->cfg.n_classes * 4)))
    return rc;

  m->plan.clear();
  Arena& A = m->arena;
  int X = 0;                                  // arena index of the current block input
  auto others = [&](int x, int (&t)[4]) { int k = 0; for (int i = 0; i < 5; ++i) if (i != x) t[k++] = i; };

  // ---- block 1
  { Op op; op.kind = OP_STATS; op.stage = 0; m->plan.push_back(op); }
  { Op op; op.kind = OP_CONV1; op.stage = 0; op.out = A.p(0); op.H = px; op.Ho = s1; op.tag = "block1_conv1";
    // output of conv1_tc_kernel as a [tiles * 149 * 149, 32] matrix: one [32 pixels x 32 channels] box per epilogue warp
    if ((rc = make_tmap(ctx, &op.tc, A.p(0), (uint64_t)B * s1 * s1, 32, 32, 32, 32))) return rc;
    m->plan.push_back(op); }
  {
    Op op; op.kind = OP_GEMM; op.stage = 1; op.tag = "block1_conv2";
    op.rows_per_tile = s1 * s1; op.blk_k = 32;
    GemmParams& g = op.gp;
    g.M = s1 * s1 * B; g.N = 64; g.K = 288; g.bn_box = 64;
    g.scale = (const float*)m->conv2.scale.p; g.shift = (const float*)m->conv2.shift.p;
    g.out = A.p(1); g.ldc = 64; g.relu = 1;
    g.conv_mode = 1; g.in_w = s1; g.in_hw = s1 * s1; g.out_w = s2; g.out_h = s2; g.out_hw = s2 * s2;
    g.a_ptr = A.p(0); g.lda = 32; g.a_rows = (long long)s1 * s1 * B;
    g.b_ptr = (const bf16*)m->conv2.w.p; g.ldb = 288;
    if ((rc = make_tmap(ctx, &op.ta, A.p(0), (uint64_t)s1 * s1 * B, 32, 32, 128, 32))) return rc;
    if ((rc = make_tmap(ctx, &op.tb, m->conv2.w.p, 64, 288, 288, 64, 32))) return rc;
    // output boxes of the epilogue warps: [1, 1, 32 pixels, 32 channels], SWIZZLE_64B staging tiles
    if ((rc = make_tmap_nhwc(ctx, &op.tc, A.p(1), (uint64_t)B, (uint64_t)s2, (uint64_t)s2, 64, 1, 32, 32, false, true))) return rc;
    op.tr = op.ta; op.tb2 = op.tb;
    op.Ho = s2; op.Wo = s2; op.Cout = 64;
    m->plan.push_back(op);
  }
  X = 1;
  int H = s2, C = 64;

  int dw_rc = BQ_OK;
  // Every op carries a tag so that bq_model_debug_stage can stop behind it: block{b}_sub, block{b}_res,
  // block{b}_sepconv{i}_dw (stand-alone depthwise), block{b}_sepconv{i} (SeparableConv after BN / ReLU), and block{b} for
  // a block output (the last sepconv of blocks 5-12 with its residual, and block14_sepconv2).
  auto add_dw = [&](const bf16* in, bf16* out, int h, int c, int relu_in, const SepWeights& sw, int stage, const std::string& tag,
                    int in_pitch = 0) {
    Op op; op.kind = OP_DW; op.stage = stage; op.in = in; op.out = out; op.H = h; op.W = h; op.C = c;
    op.relu_in = relu_in; op.dw = (const float*)sw.dw.p;
    const int CC = (c % 64 != 0) ? 56 : 64;                            // 728 = 13 x 56
    int r = make_tmap_nhwc(ctx, &op.ta, in, (uint64_t)B, (uint64_t)h, (uint64_t)h, (uint64_t)c, bq::dwp::kHalo, bq::dwp::kHalo, CC,
                           false, false, (uint64_t)in_pitch);
    if (r && !dw_rc) dw_rc = r;
    op.tag = tag;
    op.Ho = h; op.Wo = h; op.Cout = c;
    m->plan.push_back(op);
  };
  auto add_gemm = [&](const bf16* a, int rows, const PwWeights& w, bf16* out, int relu, const bf16* resid, int stage,
                      const std::string& tag, int h, int cout) -> int {
    Op op; op.stage = stage;
    int r = make_gemm(m, op, a, rows, w, out, relu, resid);
    if (r) return r;
    op.tag = tag;
    op.Ho = h; op.Wo = h; op.Cout = cout;
    m->plan.push_back(op);
    return BQ_OK;
  };
  // one SeparableConv2D `name` (+BN, optional ReLU / residual): fused entry-flow kernel for 64/128/256 -> 128/256,
  // otherwise depthwise + GEMM; the output is tagged `tag`, or `name` when tag is null
  auto add_sep = [&](const bf16* in, bf16* dw_tmp, int h, int cin, int relu_in, const SepWeights& sw, bf16* out, int relu_out,
                     const bf16* resid, int stage, const std::string& name, const char* tag, int in_pitch = 0) -> int {
    if (!in_pitch && !m->use_simt && !resid && cin % 64 == 0 && cin <= 256 && (sw.pw.cout == 128 || sw.pw.cout == 256)) {
      Op op; op.kind = OP_SEP2D; op.stage = stage;
      op.tag = tag ? tag : name;
      op.in = in; op.out = out; op.H = h; op.W = h; op.C = cin; op.Ho = h; op.Wo = h; op.Cout = sw.pw.cout;
      op.s2.n_img = B; op.s2.H = h; op.s2.W = h; op.s2.K = cin; op.s2.N = sw.pw.cout;
      op.s2.relu_in = relu_in; op.s2.relu_out = relu_out;
      op.s2.dw = (const float*)sw.dw.p; op.s2.scale = (const float*)sw.pw.scale.p; op.s2.shift = (const float*)sw.pw.shift.p;
      int r;
      if ((r = make_tmap_nhwc(ctx, &op.ta, in, (uint64_t)B, (uint64_t)h, (uint64_t)h, (uint64_t)cin, bq::sep2d::kHH, bq::sep2d::kHW, 64, false))) return r;
      if ((r = make_tmap(ctx, &op.tb, sw.pw.w.p, (uint64_t)sw.pw.cout, (uint64_t)cin, (uint64_t)cin, (uint32_t)sw.pw.cout, 64))) return r;
      // one box per epilogue warp and step: 32 channels x 16 columns x 2 patch rows, SWIZZLE_64B staging tiles
      if ((r = make_tmap_nhwc(ctx, &op.tc, out, (uint64_t)B, (uint64_t)h, (uint64_t)h, (uint64_t)sw.pw.cout, 2, bq::sep2d::kPW, 32, false, true))) return r;
      m->plan.push_back(op);
      return BQ_OK;
    }
    add_dw(in, dw_tmp, h, cin, relu_in, sw, stage, name + "_dw", in_pitch);
    return add_gemm(dw_tmp, h * h, sw.pw, out, relu_out, resid, stage, tag ? tag : name, h, sw.pw.cout);
  };
  // entry-style block with a strided 1x1 residual branch and a max-pool (blocks 2,3,4,13)
  // `padded_in` / `padded_out`: the block input / output lives in the zero-padded middle-flow layout (pitch 20), which
  // saves the two layout-conversion copies around blocks 5-12
  auto res_block = [&](int b, int cout1, int cout2, int relu_first, int stage, const bf16* padded_in = nullptr,
                       bf16* padded_out = nullptr) -> int {
    int t[4]; others(X, t);
    const int Ho = (H + 1) / 2;
    const bf16* xin = padded_in ? padded_in : A.p(X);
    const int in_pitch = padded_in ? bq::sepmid::kPitch : 0;
    const std::string pre = "block" + std::to_string(b);
    const SepWeights& s1w = *m->sep.at(pre + "_sepconv1");
    const SepWeights& s2w = *m->sep.at(pre + "_sepconv2");
    const PwWeights& rw = *m->res.at(pre + "_res");
    { Op op; op.kind = OP_SUBSAMPLE; op.stage = stage; op.in = xin; op.in_pitch = in_pitch; op.out = A.p(t[0]); op.H = H; op.W = H; op.Ho = Ho; op.Wo = Ho; op.C = C;
      op.Cout = C; op.tag = pre + "_sub"; m->plan.push_back(op); }
    int r;
    if ((r = add_gemm(A.p(t[0]), Ho * Ho, rw, A.p(t[1]), 0, nullptr, stage, pre + "_res", Ho, cout2))) return r;   // res -> t1
    if ((r = add_sep(xin, A.p(t[0]), H, C, relu_first, s1w, A.p(t[2]), 1, nullptr, stage, pre + "_sepconv1", nullptr, in_pitch))) return r;
    if ((r = add_sep(A.p(t[2]), A.p(t[0]), H, cout1, 0, s2w, A.p(t[3]), 0, nullptr, stage, pre + "_sepconv2", nullptr))) return r;
    { Op op; op.kind = OP_POOLADD; op.stage = stage; op.in = A.p(t[3]); op.in2 = A.p(t[1]); op.out = padded_out ? padded_out : A.p(X);
      op.out_pitch = padded_out ? bq::sepmid::kPitch : 0; op.padded_out = padded_out != nullptr;
      op.H = H; op.W = H; op.Ho = Ho; op.Wo = Ho; op.C = cout2; op.Cout = cout2; op.pad_top = same_pad_before(H); op.pad_left = same_pad_before(H);
      op.tag = pre; m->plan.push_back(op); }
    H = Ho; C = cout2;
    return BQ_OK;
  };
  if ((rc = res_block(2, 128, 128, 0, 2)) || (rc = res_block(3, 256, 256, 1, 2))) return rc;
  // Fused depthwise->pointwise kernel on the zero-padded flattened layout (sepmid_sm100.cuh) for the middle flow.  The
  // four buffers are dedicated to this layout: zeroed once here, and only VALID pixels are ever written, so the border
  // stays zero.  Block 4's pool+add writes its output straight into that layout and block 13 reads it from there.
  const bool mid = m->sep_mid && (H + 1) / 2 == bq::sepmid::kMap;
  auto P = [&](int i) { return (bf16*)m->midbuf[i].p; };
  if (mid) {
    using namespace bq::sepmid;
    const uint64_t rows = (uint64_t)B * kImgRows + kSlackRows;
    for (auto& b : m->midbuf) {
      if ((rc = bq_alloc(ctx, b, rows * kC * sizeof(bf16)))) return rc;
      BQ_CUDA(ctx, cudaMemset(b.p, 0, rows * kC * sizeof(bf16)));
    }
  }
  if ((rc = res_block(4, 728, 728, 1, 2, nullptr, mid ? P(0) : nullptr))) return rc;
  // ---- middle flow: 8 x (3 x (ReLU, sepconv, BN)) + identity
  int mid_out = -1;                               // padded buffer holding the output of block 12
  if (mid) {
    using namespace bq::sepmid;
    const uint64_t rows = (uint64_t)B * kImgRows + kSlackRows;
    auto add_mid = [&](int src, int dst, int res, const SepWeights& sw, int relu_in, int relu_out, const std::string& tag) -> int {
      Op op; op.kind = OP_SEPMID; op.stage = 3; op.padded_out = true;
      op.tag = tag;
      op.in = P(src); op.out = P(dst); op.in2 = res >= 0 ? P(res) : nullptr;
      op.H = kMap; op.W = kMap; op.C = kC; op.Ho = kMap; op.Wo = kMap; op.Cout = kC; op.relu_in = relu_in;
      op.sm.n_rows = B * kImgRows; op.sm.relu_out = relu_out;
      op.sm.dw = (const float*)sw.dw.p; op.sm.scale = (const float*)sw.pw.scale.p; op.sm.shift = (const float*)sw.pw.shift.p;
      op.sm.residual = op.in2;
      int r;
      if ((r = make_tmap(ctx, &op.ta, P(src), rows, kC, kC, kWinRows, 64, true))) return r;
      if ((r = make_tmap(ctx, &op.tb, sw.pw.w.p, kC, kC, kC, 128, 64))) return r;
      // 32-channel (64-byte) boxes, SWIZZLE_64B: the fragment epilogue writes stmatrix rows
      if ((r = make_tmap(ctx, &op.tc, P(dst), rows, kC, kC, kMap, 32))) return r;
      op.tr = op.tc;
      if (res >= 0 && (r = make_tmap(ctx, &op.tr, P(res), rows, kC, kC, kStepPx, 32))) return r;
      m->plan.push_back(op);
      return BQ_OK;
    };
    int x = 0;                                   // padded buffer holding the block input (= residual)
    for (int b = 5; b <= 12; ++b) {
      const std::string pre = "block" + std::to_string(b) + "_sepconv";
      const SepWeights &w1 = *m->sep.at(pre + "1"), &w2 = *m->sep.at(pre + "2"), &w3 = *m->sep.at(pre + "3");
      const std::string tag = "block" + std::to_string(b);
      const int a = (x + 1) & 3, bb = (x + 2) & 3, c = (x + 3) & 3;
      if ((rc = add_mid(x, a, -1, w1, 1, 1, pre + "1"))) return rc;
      if ((rc = add_mid(a, bb, -1, w2, 0, 1, pre + "2"))) return rc;
      if ((rc = add_mid(bb, c, x, w3, 0, 0, tag))) return rc;
      x = c;
    }
    mid_out = x;
  } else
  for (int b = 5; b <= 12; ++b) {
    int t[4]; others(X, t);
    const std::string pre = "block" + std::to_string(b) + "_sepconv";
    const SepWeights &w1 = *m->sep.at(pre + "1"), &w2 = *m->sep.at(pre + "2"), &w3 = *m->sep.at(pre + "3");
    // (the unfused path ping-pongs t0 <-> t1; the fused kernel must not write its own input, so it uses t1 -> t3 -> t2)
    const std::string tag = "block" + std::to_string(b);
    if ((rc = add_sep(A.p(X), A.p(t[0]), H, C, 1, w1, A.p(t[1]), 1, nullptr, 3, pre + "1", nullptr))) return rc;
    if ((rc = add_sep(A.p(t[1]), A.p(t[0]), H, C, 0, w2, A.p(t[3]), 1, nullptr, 3, pre + "2", nullptr))) return rc;
    if ((rc = add_sep(A.p(t[3]), A.p(t[0]), H, C, 0, w3, A.p(t[2]), 0, A.p(X), 3, pre + "3", tag.c_str()))) return rc;
    X = t[2];
  }
  // ---- exit flow
  if ((rc = res_block(13, 728, 1024, 1, 4, mid_out >= 0 ? P(mid_out) : nullptr))) return rc;
  {
    int t[4]; others(X, t);
    const SepWeights &w1 = *m->sep.at("block14_sepconv1"), &w2 = *m->sep.at("block14_sepconv2");
    add_dw(A.p(X), A.p(t[0]), H, C, 0, w1, 4, "block14_sepconv1_dw");
    if ((rc = add_gemm(A.p(t[0]), H * H, w1.pw, A.p(t[1]), 1, nullptr, 4, "block14_sepconv1", H, 1536))) return rc;
    add_dw(A.p(t[1]), A.p(t[0]), H, 1536, 0, w2, 4, "block14_sepconv2_dw");
    if ((rc = add_gemm(A.p(t[0]), H * H, w2.pw, A.p(t[2]), 1, nullptr, 4, "block14", H, kFeatures))) return rc;
    Op op; op.kind = OP_GAP; op.stage = 4; op.in = A.p(t[2]); op.H = H; op.W = H; op.C = kFeatures; m->plan.push_back(op);
  }
  return dw_rc;
}

int run_op(bq_model* m, Op& op, int nb, int64_t out_off = 0) {
  bq_ctx* ctx = m->ctx;
  const int px = m->px;
  auto grid1d = [&](int64_t total) {
    int64_t g = (total + 255) / 256;
    const int64_t cap = (int64_t)ctx->num_sms * 32;
    return (int)(g > cap ? cap : (g < 1 ? 1 : g));
  };
  const double act = 2.0;   // bytes per bf16 activation element
  switch (op.kind) {
    case OP_STATS: {
      if (m->input_f32) return BQ_OK;              // standardised by the caller
      KScope ks(m, BQ_K_STATS, 0, (double)nb * px * px * 3);
      bq::tile_stats_kernel<<<nb, 512, 0, ctx->stream>>>(m->tiles_src, (int64_t)px * px * 3,
                                                        (float*)m->mean.p, (float*)m->inv_std.p, (const float*)m->conv1_sumw.p,
                                                        (const float*)m->conv1_scale.p, (const float*)m->conv1_shift.p,
                                                        (float*)m->conv1_affine.p, (float*)m->conv1_m0.p);
      break;
    }
    case OP_CONV1: {
      KScope ks(m, BQ_K_CONV1, 2.0 * nb * op.Ho * op.Ho * 27 * 32, (double)nb * px * px * 3 + act * nb * op.Ho * op.Ho * 32);
      dim3 grid((op.Ho + bq::kC1Tile - 1) / bq::kC1Tile, (op.Ho + bq::kC1Tile - 1) / bq::kC1Tile, nb);
      if (!m->input_f32 && !m->use_simt && px == bq::conv1tc::kIn) {
        // raw uint8 pixels on the tensor cores, standardisation applied behind the convolution (conv1_sm100.cuh)
        bq::conv1tc::Conv1Params cp;
        cp.tiles = m->tiles_src; cp.affine = (const float*)m->conv1_affine.p; cp.m0 = (const float*)m->conv1_m0.p;
        cp.w = (const bf16*)m->conv1_wtc.p; cp.out = op.out; cp.n_img = nb;
        const int items = nb * bq::conv1tc::kItemsPerImg;
        const int g1 = items < 2 * ctx->num_sms ? items : 2 * ctx->num_sms;
        bq::conv1tc::conv1_tc_kernel<<<g1, bq::conv1tc::kThreads, bq::conv1tc::kSmem, ctx->stream>>>(op.tc, cp);
      } else if (m->input_f32)
        bq::conv1_kernel<float><<<grid, 256, 0, ctx->stream>>>((const float*)m->tiles_src, (const float*)m->mean.p,
                                                              (const float*)m->inv_std.p, (const float*)m->conv1_w.p,
                                                              (const float*)m->conv1_scale.p, (const float*)m->conv1_shift.p,
                                                              op.out, px, op.Ho);
      else
        bq::conv1_kernel<uint8_t><<<grid, 256, 0, ctx->stream>>>(m->tiles_src, (const float*)m->mean.p,
                                                                (const float*)m->inv_std.p, (const float*)m->conv1_w.p,
                                                                (const float*)m->conv1_scale.p, (const float*)m->conv1_shift.p,
                                                                op.out, px, op.Ho);
      break;
    }
    case OP_GEMM: {
      GemmParams g = op.gp;
      g.M = op.rows_per_tile * nb;
      g.a_rows = (long long)op.rows_per_tile * m->max_batch;
      const double rows_out = g.conv_mode ? (double)nb * g.out_hw : (double)g.M;
      const double kin = g.conv_mode ? g.K / 9 : g.K;
      KScope ks(m, g.conv_mode ? BQ_K_GEMM_CONV2 : BQ_K_GEMM_PW, 2.0 * rows_out * g.N * g.K,
                act * ((double)g.M * kin + rows_out * g.N * (g.residual ? 2 : 1) + (double)g.N * g.K));
      return launch_gemm(m, g, op.ta, op.tb, op.tc, op.tr, op.blk_k, g.conv_mode ? nullptr : &op.tb2);
    }
    case OP_DW: {
      KScope ks(m, BQ_K_DW, 2.0 * 9 * nb * op.H * op.W * op.C, 2 * act * nb * op.H * op.W * op.C);
      const int CC = (op.C % 64 != 0) ? 56 : 64;                        // 728 = 13 x 56
      const int tiles = (op.H + bq::dwp::kTile - 1) / bq::dwp::kTile;
      const int64_t items = (int64_t)nb * tiles * tiles * (op.C / CC);
      const int grid = (int)std::min<int64_t>(items, ctx->num_sms);
#define BQ_DWP_LAUNCH(RELU, CCV)                                                                              \
  bq::dwp::depthwise3x3_pipe_kernel<RELU, CCV><<<grid, bq::dwp::kThreads, bq::dwp::kSmem, ctx->stream>>>(    \
      op.ta, op.dw, op.out, nb, op.H, op.W, op.C, tiles)
      if (CC == 56) { if (op.relu_in) BQ_DWP_LAUNCH(true, 56); else BQ_DWP_LAUNCH(false, 56); }
      else          { if (op.relu_in) BQ_DWP_LAUNCH(true, 64); else BQ_DWP_LAUNCH(false, 64); }
#undef BQ_DWP_LAUNCH
      break;
    }
    case OP_POOLADD: {
      KScope ks(m, BQ_K_POOLADD, 0, act * nb * op.C * ((double)op.H * op.W + 2.0 * op.Ho * op.Wo));
      bq::maxpool_add_kernel<<<grid1d((int64_t)nb * op.Ho * op.Wo * (op.C / 8)), 256, 0, ctx->stream>>>(
          op.in, op.in2, op.out + out_off, nb, op.H, op.W, op.Ho, op.Wo, op.C, op.pad_top, op.pad_left, op.out_pitch);
      break;
    }
    case OP_SUBSAMPLE: {
      KScope ks(m, BQ_K_SUBSAMPLE, 0, 2 * act * nb * op.Ho * op.Wo * op.C);
      bq::subsample2_kernel<<<grid1d((int64_t)nb * op.Ho * op.Wo * (op.C / 8)), 256, 0, ctx->stream>>>(
          op.in, op.out, nb, op.H, op.W, op.Ho, op.Wo, op.C, op.in_pitch);
      break;
    }
    case OP_SEP2D: {
      bq::sep2d::Sep2dParams s2 = op.s2;
      s2.n_img = nb;
      const int items = nb * ((op.H + bq::sep2d::kPH - 1) / bq::sep2d::kPH) * ((op.W + bq::sep2d::kPW - 1) / bq::sep2d::kPW);
      const int grid = items < ctx->num_sms ? items : ctx->num_sms;
      const double px_n = (double)nb * op.H * op.W;
      KScope ks(m, BQ_K_SEP_FUSED, 2.0 * px_n * s2.K * (s2.N + 9.0), act * px_n * (s2.K + s2.N));
      const int smem2d = bq::sep2d::smem_bytes(s2.N);
      if (s2.relu_in)
        bq::sep2d::sepconv2d_fused_kernel<true><<<grid, bq::sep2d::kThreads, smem2d, ctx->stream>>>(op.ta, op.tb, op.tc, s2);
      else
        bq::sep2d::sepconv2d_fused_kernel<false><<<grid, bq::sep2d::kThreads, smem2d, ctx->stream>>>(op.ta, op.tb, op.tc, s2);
      break;
    }
    case OP_SEPMID: {
      bq::sepmid::SepMidParams sm = op.sm;
      sm.n_rows = nb * bq::sepmid::kImgRows;
      const int items = (sm.n_rows + bq::sepmid::kItemPx - 1) / bq::sepmid::kItemPx;
      const int clusters = items < ctx->num_sms / 2 ? items : ctx->num_sms / 2;
      const double px_n = (double)nb * op.H * op.W;
      KScope ks(m, BQ_K_SEP_MID, 2.0 * px_n * op.C * (op.C + 9.0), act * px_n * op.C * (sm.residual ? 3.0 : 2.0));
      if (op.relu_in)
        bq::sepmid::sepconv_mid_kernel<true><<<2 * clusters, bq::sepmid::kThreads, bq::sepmid::kSmem, ctx->stream>>>(op.ta, op.tb, op.tc, op.tr, sm);
      else
        bq::sepmid::sepconv_mid_kernel<false><<<2 * clusters, bq::sepmid::kThreads, bq::sepmid::kSmem, ctx->stream>>>(op.ta, op.tb, op.tc, op.tr, sm);
      break;
    }
    case OP_GAP: {
      KScope ks(m, BQ_K_GAP, 0, act * nb * op.H * op.W * op.C + 6.0 * nb * op.C);
      bq::gap_kernel<<<grid1d((int64_t)nb * op.C), 256, 0, ctx->stream>>>(op.in, (float*)m->feat.p,
                                                                           (bf16*)m->feat_bf16.p, nb, op.H * op.W, op.C);
      break;
    }
  }
  BQ_LAUNCH_CHECK(ctx);
  return BQ_OK;
}

int stage_tiles(bq_model* m, const uint8_t* tiles, int nb) {
  bq_ctx* ctx = m->ctx;
  const size_t bytes = (size_t)nb * m->px * m->px * 3;
  BQ_CUDA(ctx, cudaMemcpyAsync(m->tiles_dev.p, tiles, bytes, cudaMemcpyDefault, ctx->stream));
  m->tiles_src = (const uint8_t*)m->tiles_dev.p;
  return BQ_OK;
}

// One micro-batch through the plan as plain stream launches (profiling, debug stops, partial micro-batches).
int run_backbone(bq_model* m, int nb, const std::string* stop_tag, const Op** stopped) {
  int cur_stage = -1;
  for (size_t i = 0; i < m->plan.size(); ++i) {
    Op& op = m->plan[i];
    if (m->profiling && op.stage != cur_stage) {
      cudaEventRecord(m->ev[op.stage], m->ctx->stream);
      cur_stage = op.stage;
    }
    int rc = run_op(m, op, nb, 0);
    if (rc) return rc;
    if (stop_tag && op.tag == *stop_tag) { if (stopped) *stopped = &op; return BQ_OK; }
  }
  if (m->profiling) cudaEventRecord(m->ev[5], m->ctx->stream);
  return BQ_OK;
}

// Full micro-batch, no profiling, no debug stop: stats + conv1 eagerly (they read the caller's tile pointer, which moves
// from micro-batch to micro-batch), everything after them as one graph replay.
int run_backbone_graphed(bq_model* m, int nb) {
  bq_ctx* ctx = m->ctx;
  size_t first = 0;
  while (first < m->plan.size() && (m->plan[first].kind == OP_STATS || m->plan[first].kind == OP_CONV1)) ++first;
  const bool ok = m->use_graph && !m->profiling && nb == m->max_batch && first > 0 && first < m->plan.size();
  if (!ok) return run_backbone(m, nb, nullptr, nullptr);
  int rc;
  for (size_t i = 0; i < first; ++i)
    if ((rc = run_op(m, m->plan[i], nb, 0))) return rc;
  if (!m->backbone_graph) {
    const int64_t before = ctx->launches;
    cudaGraph_t graph = nullptr;
    BQ_CUDA(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    rc = BQ_OK;
    for (size_t i = first; i < m->plan.size() && rc == BQ_OK; ++i) rc = run_op(m, m->plan[i], nb, 0);
    cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) return bq_fail(ctx, BQ_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
    m->graph_kernels = ctx->launches - before;
    ctx->launches = before;
    e = cudaGraphInstantiate(&m->backbone_graph, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { m->backbone_graph = nullptr; return bq_fail(ctx, BQ_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
  }
  BQ_CUDA(ctx, cudaGraphLaunch(m->backbone_graph, ctx->stream));
  ctx->launches += m->graph_kernels;
  return BQ_OK;
}

// (re)build head GEMM descriptors for T samples
int prepare_head(bq_model* m, int T) {
  bq_ctx* ctx = m->ctx;
  if (m->head_T == T) return BQ_OK;
  const int B = m->max_batch, Wd = m->cfg.hidden_width, Hn = m->cfg.hidden_layers;
  int rc;
  size_t rows = (size_t)B * T;
  if (rows < (size_t)m->head_batch) rows = (size_t)m->head_batch;
  if (T > m->head_T_cap) {
    BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t hrows = (m->sites & 1) ? (size_t)(m->head_batch > B ? m->head_batch : B) * T : rows;
    for (auto& h : m->h_act) { h.release(); if ((rc = bq_alloc(ctx, h, hrows * Wd * 2 + 1024))) return rc; }
    m->a2.release();
    if ((rc = bq_alloc(ctx, m->a2, rows * Wd * 2 + 1024))) return rc;
    m->a0.release();
    if ((m->sites & 1) && (rc = bq_alloc(ctx, m->a0, (size_t)B * T * kFeatures * 2 + 1024))) return rc;
    m->head_T_cap = T;
  }
  m->head_gemms.clear();
  m->head_gemms.resize(Hn);
  const float inv_keep = 1.0f / (1.0f - m->cfg.dropout);
  for (int i = 0; i < Hn; ++i) {
    Op op;
    const PwWeights& w = *m->hidden[i];
    // layer 0: A = pooled features [B, 2048] -> h_act[0] [B, Wd]; layer i>0: A = masked operand [B*T, Wd]
    const bool site0 = (m->sites & 1) != 0;
    const bf16* a = i == 0 ? (site0 ? (const bf16*)m->a0.p : (const bf16*)m->feat_bf16.p) : (const bf16*)m->a2.p;
    bf16* out = (bf16*)m->h_act[i & 1].p;
    m->max_batch = (i == 0 && !site0) ? B : B * T;   // make_gemm sizes M = rows_per_tile * max_batch
    const float alpha = (m->sites >> i) & 1 ? inv_keep : 1.0f;        // 1/(1-p) behind an enabled site
    rc = make_gemm(m, op, a, 1, w, out, 1, nullptr, alpha);
    m->max_batch = B;
    if (rc) return rc;
    if (i == 0) {   // layer-0 output map spans the whole head batch: micro-batches land at their row offset
      if ((rc = make_tmap(ctx, &op.tc, out, (uint64_t)(m->head_batch > B ? m->head_batch : B) * (site0 ? T : 1), (uint64_t)w.cout,
                          (uint64_t)w.cout, 128, 64)))
        return rc;
    }
    m->head_gemms[i].gp = op.gp;
    m->head_gemms[i].ta = op.ta;
    m->head_gemms[i].tb = op.tb;
    m->head_gemms[i].tc = op.tc;
    m->head_gemms[i].tb2 = op.tb2;
  }
  m->head_T = T;
  return BQ_OK;
}

// phase 1 (per micro-batch): hidden_0 on the pooled features, written at row `h1_off` of the head buffer.
// phase 2 (`n_head` > 0): the dropout-bearing layers for the n_head tiles accumulated so far.
int run_head(bq_model* m, int nb, int T, uint64_t seed, uint64_t tile_base, const uint8_t* masks_dev, int h1_off = 0,
             int n_head = -1) {
  bq_ctx* ctx = m->ctx;
  const int Wd = m->cfg.hidden_width, Hn = m->cfg.hidden_layers, NC = m->cfg.n_classes;
  const uint32_t thresh = (uint32_t)floor((double)m->cfg.dropout * 4294967296.0);
  int rc = prepare_head(m, T);
  if (rc) return rc;
  auto grid1d = [&](int64_t total) {
    int64_t g = (total + 255) / 256;
    const int64_t cap = (int64_t)ctx->num_sms * 32;
    return (int)(g > cap ? cap : (g < 1 ? 1 : g));
  };
  if (Hn != 2 || Wd > bq::head::kHMaxW || Wd % 64) return bq_fail(ctx, BQ_ERR_ARG, "the fused MC-dropout head needs 2 hidden layers of width <= 1024 (hp.py:13,21)");
  if (nb > 0) {
    // ---- hidden_0 of this micro-batch (GEMM kernel), written at row h1_off of the head buffer
    auto& hg = m->head_gemms[0];
    GemmParams g = hg.gp;
    if (m->sites & 1) {
      // dropout on the pooled features: one masked copy of the feature row per (tile, sample), so hidden_0 is per sample
      KScope ks(m, BQ_K_MC_EXPAND, 0, 2.0 * nb * kFeatures + 2.0 * nb * T * kFeatures);
      bq::mc_expand_kernel<<<grid1d((int64_t)nb * T * (kFeatures / 4)), 256, 0, ctx->stream>>>(
          (const bf16*)m->feat_bf16.p, (bf16*)m->a0.p, nb, T, kFeatures, seed, tile_base, 0, thresh, masks_dev, m->n_sites,
          m->slot[0], m->mask_w);
      BQ_LAUNCH_CHECK(ctx);
      g.M = nb * T;
      g.out_row_off = h1_off * T;
    } else {
      g.M = nb;
      g.out_row_off = h1_off;
    }
    KScope ks(m, BQ_K_HEAD_GEMM, 2.0 * g.M * g.N * g.K, 2.0 * ((double)g.M * g.K + (double)g.M * g.N + (double)g.N * g.K));
    if ((rc = launch_gemm(m, g, hg.ta, hg.tb, hg.tc, hg.tc, 64, &hg.tb2))) return rc;
  }
  if (n_head < 0) n_head = nb;
  if (n_head == 0) return BQ_OK;
  nb = n_head;
  // ---- ONE kernel: Philox masks -> hidden_1 (tcgen05) -> bias/ReLU -> mask -> prelogits -> softmax -> mean/std over T
  bq::head::HeadParams hp;
  hp.h1 = (const bf16*)m->h_act[0].p;
  hp.b2 = (const float*)m->hidden[1]->shift.p;
  hp.w3 = (const float*)m->w3.p;
  hp.b3 = (const float*)m->b3.p;
  hp.mean = (float*)m->out_mean.p;
  hp.stdv = (float*)m->out_std.p;
  hp.masks = masks_dev;
  hp.n = nb; hp.T = T; hp.W = Wd; hp.C = NC;
  hp.n_sites = m->n_sites; hp.slot1 = m->slot[1]; hp.slot2 = m->slot[2];
  hp.mask_w = m->mask_w;
  hp.w2_box = m->head_gemms[1].gp.bn_box;          // the box rows the W2 tensor map was built with
  hp.h1_per_sample = (m->sites & 1) ? 1 : 0;
  hp.inv_keep = 1.0f / (1.0f - m->cfg.dropout);
  hp.inv_keep1 = (m->sites & 2) ? hp.inv_keep : 1.0f;
  hp.inv_keep2 = (m->sites & 4) ? hp.inv_keep : 1.0f;
  hp.thresh = thresh;
  hp.seed = seed; hp.tile_base = tile_base;
  const int groups = (nb + 3) / 4;
  const int grid = groups < ctx->num_sms ? groups : ctx->num_sms;
  KScope ks(m, BQ_K_HEAD_FUSED, 2.0 * nb * T * Wd * (Wd + NC), 2.0 * nb * Wd + 2.0 * Wd * Wd + 8.0 * nb * NC);
  bq::head::mc_head_fused_kernel<<<grid, bq::head::kHThreads, bq::head::HeadSmem::kTotal, ctx->stream>>>(m->head_gemms[1].tb, hp);
  BQ_LAUNCH_CHECK(ctx);
  return BQ_OK;
}

__global__ void bf16_to_f32_kernel(const bf16* in, float* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = __bfloat162float(in[i]);
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int bq_model_create(bq_ctx* ctx, const bq_model_config* cfg, bq_model** out) {
  if (!ctx) return BQ_ERR_ARG;
  if (!cfg || !out) return bq_fail(ctx, BQ_ERR_ARG, "bq_model_create: null argument");
  if (cfg->tile_px != 299) return bq_fail(ctx, BQ_ERR_ARG, "tile_px must be 299 (hp.py:5), got %d", cfg->tile_px);
  if (cfg->hidden_layers != 2) return bq_fail(ctx, BQ_ERR_ARG, "hidden_layers must be 2 (hp.py:21), got %d", cfg->hidden_layers);
  if (cfg->hidden_width <= 0 || cfg->hidden_width % 64) return bq_fail(ctx, BQ_ERR_ARG, "hidden_width must be a positive multiple of 64");
  if (cfg->hidden_width > bq::head::kHMaxW) return bq_fail(ctx, BQ_ERR_ARG, "the fused MC-dropout head needs 2 hidden layers of width <= 1024 (hp.py:13,21)");
  if (cfg->n_classes < 2 || cfg->n_classes > bq::kMaxClasses) return bq_fail(ctx, BQ_ERR_ARG, "n_classes must be in [2,8]");
  if (!(cfg->dropout >= 0.f && cfg->dropout < 1.f)) return bq_fail(ctx, BQ_ERR_ARG, "dropout must be in [0,1)");
  if (cfg->max_batch < 1 || cfg->max_batch > 512) return bq_fail(ctx, BQ_ERR_ARG, "max_batch must be in [1,512]");
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  bq_model* m = new bq_model();
  m->ctx = ctx;
  m->cfg = *cfg;
  m->max_batch = cfg->max_batch;
  m->px = cfg->tile_px;
  m->sites = cfg->dropout_sites ? cfg->dropout_sites : 6;
  if (m->sites & ~7) { delete m; return bq_fail(ctx, BQ_ERR_ARG, "dropout_sites must be a bitmask of sites 0..2"); }
  m->n_sites = 0;
  for (int i = 0; i < 3; ++i) m->slot[i] = (m->sites >> i) & 1 ? m->n_sites++ : -1;
  m->mask_w = (m->sites & 1) ? kFeatures : cfg->hidden_width;
  // Debug switches (never the default; each is exercised by a test): BQ_GEMM=simt runs every GEMM-shaped op on a plain
  // CUDA-core kernel, BQ_GRAPH=off launches the backbone op by op, BQ_SEPMID=off runs the 728-wide middle flow as
  // stand-alone depthwise + pointwise-GEMM kernels instead of the fused kernel.
  const char* g = getenv("BQ_GEMM");
  m->use_simt = g && strcmp(g, "simt") == 0;
  const char* gr = getenv("BQ_GRAPH");
  m->use_graph = !(gr && strcmp(gr, "off") == 0);
  const char* smid = getenv("BQ_SEPMID");
  m->sep_mid = !(smid && strcmp(smid, "off") == 0) && !m->use_simt;
  using namespace bq::sm100;
  cudaFuncSetAttribute(gemm_tcgen05_2cta_kernel<k2Stages>, cudaFuncAttributeMaxDynamicSharedMemorySize, SmemPlan2<k2Stages>::kTotal);
  cudaFuncSetAttribute(gemm_tcgen05_2cta_kernel<k2Stages + 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SmemPlan2<k2Stages + 1>::kTotalNoRes);
  cudaFuncSetAttribute(conv3x3_is_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kC2Smem);
  cudaFuncSetAttribute(bq::conv1tc::conv1_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::conv1tc::kSmem);
  cudaFuncSetAttribute(bq::head::mc_head_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::head::HeadSmem::kTotal);
  cudaFuncSetAttribute(bq::sep2d::sepconv2d_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::sep2d::smem_bytes(256));
  cudaFuncSetAttribute(bq::sep2d::sepconv2d_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::sep2d::smem_bytes(256));
  cudaFuncSetAttribute(bq::sepmid::sepconv_mid_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::sepmid::kSmem);
  cudaFuncSetAttribute(bq::sepmid::sepconv_mid_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::sepmid::kSmem);
  cudaFuncSetAttribute(bq::dwp::depthwise3x3_pipe_kernel<true, 56>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::dwp::kSmem);
  cudaFuncSetAttribute(bq::dwp::depthwise3x3_pipe_kernel<false, 56>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::dwp::kSmem);
  cudaFuncSetAttribute(bq::dwp::depthwise3x3_pipe_kernel<true, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::dwp::kSmem);
  cudaFuncSetAttribute(bq::dwp::depthwise3x3_pipe_kernel<false, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, bq::dwp::kSmem);
  for (auto& e : m->ev) cudaEventCreate(&e);
  cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking);
  for (int i = 0; i < 2; ++i) {
    cudaEventCreateWithFlags(&m->copied[i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&m->consumed[i], cudaEventDisableTiming);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { delete m; return bq_fail(ctx, BQ_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e)); }
  *out = m;
  return BQ_OK;
}

void bq_model_destroy(bq_model* m) {
  if (!m) return;
  cudaSetDevice(m->ctx->device);
  cudaStreamSynchronize(m->ctx->stream);
  if (m->backbone_graph) cudaGraphExecDestroy(m->backbone_graph);
  for (auto& e : m->ev) if (e) cudaEventDestroy(e);
  for (auto& e : m->kev) cudaEventDestroy(e);
  if (m->copy_stream) { cudaStreamSynchronize(m->copy_stream); cudaStreamDestroy(m->copy_stream); }
  for (int i = 0; i < 2; ++i) { if (m->copied[i]) cudaEventDestroy(m->copied[i]); if (m->consumed[i]) cudaEventDestroy(m->consumed[i]); }
  delete m->jpeg;
  delete m->png;
  delete m;
}

int bq_model_load_weights(bq_model* m, const bq_named_tensor* tensors, int32_t n_tensors) {
  if (!m) return BQ_ERR_ARG;
  bq_ctx* ctx = m->ctx;
  if (!tensors || n_tensors <= 0) return bq_fail(ctx, BQ_ERR_ARG, "bq_model_load_weights: no tensors");
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  if (m->backbone_graph) { cudaGraphExecDestroy(m->backbone_graph); m->backbone_graph = nullptr; }   // the plan is rebuilt below
  TensorIndex ti;
  for (int i = 0; i < n_tensors; ++i)
    if (tensors[i].name) ti.by_name[tensors[i].name] = &tensors[i];
  int rc;
  // block1_conv1: fp32 [3,3,3,32] used as-is ([27][32]) by the fused decode/standardise/conv kernel
  {
    const bq_named_tensor* k;
    if ((rc = need(ctx, ti, "block1_conv1/kernel", {3, 3, 3, 32}, &k))) return rc;
    if ((rc = upload(ctx, m->conv1_w, k->data, 27 * 32 * 4))) return rc;
    {
      // conv1_tc_kernel: w = hi + mid + lo with three bf16 terms (3 x 8 significand bits = fp32's 24, each residual is
      // exact), rows = part * 32 + channel, K = tap * 3 + ci padded 27 -> 32; and the per-channel tap sum that carries
      // the per-image mean through the convolution
      std::vector<uint16_t> wt((size_t)96 * 32, 0);
      std::vector<float> sumw(32);
      for (int c = 0; c < 32; ++c) {
        double acc = 0.0;
        for (int kk = 0; kk < 27; ++kk) {
          const float w = k->data[(size_t)kk * 32 + c];
          acc += (double)w;
          float rem = w;
          for (int part = 0; part < 3; ++part) {
            const uint16_t b = f32_to_bf16_rne(rem);
            const uint32_t u = (uint32_t)b << 16;
            float bf;
            memcpy(&bf, &u, 4);
            wt[(size_t)(part * 32 + c) * 32 + kk] = b;
            rem -= bf;
          }
        }
        sumw[c] = (float)acc;
      }
      if ((rc = upload(ctx, m->conv1_wtc, wt.data(), wt.size() * 2)) || (rc = upload(ctx, m->conv1_sumw, sumw.data(), 32 * 4))) return rc;
    }
    PwWeights tmp;
    if ((rc = load_bn(ctx, ti, "block1_conv1_bn", 32, tmp))) return rc;
    m->conv1_scale.release(); m->conv1_shift.release();
    std::swap(m->conv1_scale.p, tmp.scale.p); std::swap(m->conv1_scale.bytes, tmp.scale.bytes); std::swap(m->conv1_scale.owned, tmp.scale.owned);
    std::swap(m->conv1_shift.p, tmp.shift.p); std::swap(m->conv1_shift.bytes, tmp.shift.bytes); std::swap(m->conv1_shift.owned, tmp.shift.owned);
  }
  if ((rc = load_conv_gemm(ctx, ti, "block1_conv2", "kernel", 3, 32, 64, m->conv2))) return rc;
  auto load_sep = [&](const std::string& name, int cin, int cout) -> int {
    std::unique_ptr<SepWeights> s(new SepWeights());
    const bq_named_tensor* d;
    int r;
    if ((r = need(ctx, ti, name + "/depthwise_kernel", {3, 3, cin, 1}, &d))) return r;
    {
      // depthwise taps are rounded to bf16 (what a bf16 model stores) and held widened to fp32 for the FFMA2 producers
      std::vector<float> dwr((size_t)9 * cin);
      for (size_t i = 0; i < dwr.size(); ++i) {
        const uint32_t u = (uint32_t)f32_to_bf16_rne(d->data[i]) << 16;
        memcpy(&dwr[i], &u, 4);
      }
      if ((r = upload(ctx, s->dw, dwr.data(), dwr.size() * 4))) return r;
    }
    if ((r = load_conv_gemm(ctx, ti, name, "pointwise_kernel", 1, cin, cout, s->pw))) return r;
    m->sep[name] = std::move(s);
    return BQ_OK;
  };
  auto load_res = [&](const std::string& name, int cin, int cout) -> int {
    std::unique_ptr<PwWeights> w(new PwWeights());
    int r = load_conv_gemm(ctx, ti, name, "kernel", 1, cin, cout, *w);
    if (r) return r;
    m->res[name] = std::move(w);
    return BQ_OK;
  };
  const int entry[3][3] = {{2, 64, 128}, {3, 128, 256}, {4, 256, 728}};
  for (auto& e : entry) {
    const std::string b = "block" + std::to_string(e[0]);
    if ((rc = load_res(b + "_res", e[1], e[2])) || (rc = load_sep(b + "_sepconv1", e[1], e[2])) ||
        (rc = load_sep(b + "_sepconv2", e[2], e[2])))
      return rc;
  }
  for (int b = 5; b <= 12; ++b)
    for (int i = 1; i <= 3; ++i)
      if ((rc = load_sep("block" + std::to_string(b) + "_sepconv" + std::to_string(i), 728, 728))) return rc;
  if ((rc = load_res("block13_res", 728, 1024)) || (rc = load_sep("block13_sepconv1", 728, 728)) ||
      (rc = load_sep("block13_sepconv2", 728, 1024)) || (rc = load_sep("block14_sepconv1", 1024, 1536)) ||
      (rc = load_sep("block14_sepconv2", 1536, 2048)))
    return rc;
  // head
  m->hidden.clear();
  int cin = kFeatures;
  for (int i = 0; i < m->cfg.hidden_layers; ++i) {
    std::unique_ptr<PwWeights> w(new PwWeights());
    if ((rc = load_dense(ctx, ti, "hidden_" + std::to_string(i), cin, m->cfg.hidden_width, *w))) return rc;
    m->hidden.push_back(std::move(w));
    cin = m->cfg.hidden_width;
  }
  {
    const bq_named_tensor *k, *b;
    if ((rc = need(ctx, ti, "prelogits/kernel", {cin, m->cfg.n_classes}, &k)) ||
        (rc = need(ctx, ti, "prelogits/bias", {m->cfg.n_classes}, &b)))
      return rc;
    if ((rc = upload(ctx, m->w3, k->data, (size_t)cin * m->cfg.n_classes * 4)) ||
        (rc = upload(ctx, m->b3, b->data, m->cfg.n_classes * 4)))
      return rc;
  }
  if ((rc = build_plan(m))) return rc;
  m->head_T = -1;
  m->weights_loaded = true;
  return BQ_OK;
}

// Input of predict_impl: decoded pixels (enc == NULL), or n compressed files back to back with n + 1 host byte offsets,
// decoded through the format state `enc`.
static int predict_impl(bq_model* m, const uint8_t* tiles, bool f32_input, bq_encoded* enc, const int64_t* offsets,
                        int64_t n, int32_t T, uint64_t seed, uint64_t tile_index_base, const uint8_t* masks, float* mean,
                        float* std, float* features);

int bq_predict_uq(bq_model* m, const uint8_t* tiles, int64_t n, int32_t T, uint64_t seed, uint64_t tile_index_base,
                  const uint8_t* masks, float* mean, float* std, float* features) {
  return predict_impl(m, tiles, false, nullptr, nullptr, n, T, seed, tile_index_base, masks, mean, std, features);
}

int bq_predict_uq_jpeg(bq_model* m, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t T, uint64_t seed,
                       uint64_t tile_index_base, const uint8_t* masks, float* mean, float* std, float* features) {
  return predict_impl(m, data, false, m ? bq_jpeg_state(m->jpeg) : nullptr, offsets, n, T, seed, tile_index_base, masks,
                      mean, std, features);
}

int bq_predict_uq_png(bq_model* m, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t T, uint64_t seed,
                      uint64_t tile_index_base, const uint8_t* masks, float* mean, float* std, float* features) {
  return predict_impl(m, data, false, m ? bq_png_state(m->png) : nullptr, offsets, n, T, seed, tile_index_base, masks,
                      mean, std, features);
}

int bq_predict_uq_standardized(bq_model* m, const float* tiles, int64_t n, int32_t T, uint64_t seed, uint64_t tile_index_base,
                               const uint8_t* masks, float* mean, float* std, float* features) {
  if (!m) return BQ_ERR_ARG;
  m->input_f32 = true;
  const int rc = predict_impl(m, (const uint8_t*)tiles, true, nullptr, nullptr, n, T, seed, tile_index_base,
                              masks, mean, std, features);
  m->input_f32 = false;
  return rc;
}

static int predict_impl(bq_model* m, const uint8_t* tiles, bool f32_input, bq_encoded* enc, const int64_t* offsets,
                        int64_t n, int32_t T, uint64_t seed, uint64_t tile_index_base, const uint8_t* masks, float* mean,
                        float* std, float* features) {
  if (!m) return BQ_ERR_ARG;
  bq_ctx* ctx = m->ctx;
  if (enc && n > 0 && !offsets)
    return bq_fail(ctx, BQ_ERR_ARG, "bq_predict_uq_%s: offsets must not be NULL", enc->api().c_str());
  if (!m->weights_loaded) return bq_fail(ctx, BQ_ERR_STATE, "bq_predict_uq: weights not loaded");
  if (n < 0 || T < 1 || T > 4096 || (n > 0 && (!tiles || !mean || !std)))
    return bq_fail(ctx, BQ_ERR_ARG, "bq_predict_uq: bad argument");
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  const int B = m->max_batch, NC = m->cfg.n_classes, Wd = m->cfg.hidden_width, Hn = m->cfg.hidden_layers;
  const size_t tile_bytes = (size_t)m->px * m->px * 3 * (f32_input ? sizeof(float) : 1);
  const size_t mask_per_tile = (size_t)T * m->n_sites * m->mask_w;
  const bool masks_on_dev = masks && bq_is_device_ptr(masks);
  if (masks && !masks_on_dev) {
    int rc = bq_alloc(ctx, m->masks_dev, (size_t)m->head_batch * mask_per_tile);
    if (rc) return rc;
  }
  int64_t head_start = 0;      // first tile of the head batch being accumulated
  int head_count = 0;
  if (m->profiling) for (auto& s : m->stage_ms) s = 0.f;
  if (m->profiling == 2)
    for (int k = 0; k < BQ_PROFILE_KINDS; ++k) { m->k_ms[k] = m->k_flops[k] = m->k_bytes[k] = 0; m->k_launches[k] = 0; }
  // Host tiles: double-buffered staging, the H2D copy of micro-batch i+1 runs on its own stream while the
  // backbone of micro-batch i computes.  Device tiles are read in place.  Compressed (JPEG / PNG) tiles always take
  // the staged route: micro-batch i + 1's descriptors (and its compressed bytes, unless they are device memory, which
  // is read in place) go up on the copy stream, and micro-batch i is decoded on the ctx stream into tiles_dev.
  const bool compressed = enc != nullptr;
  if (compressed) {
    const int rcj = enc->prepare(ctx, tiles, offsets, n, m->px, B, nullptr);
    if (rcj) return rcj;
  }
  const bool tiles_on_dev = !compressed && bq_is_device_ptr(tiles);
  if (f32_input && !tiles_on_dev) {
    const int64_t cap = n < B ? n : B;                      // the interface is usually called tile by tile (results.py:249-257)
    for (auto& b : m->tiles_f32) { int rcf = bq_alloc(ctx, b, (size_t)cap * tile_bytes + 64); if (rcf) return rcf; }
  }
  uint8_t* stage[2] = {(uint8_t*)(f32_input ? m->tiles_f32[0].p : m->tiles_dev.p), (uint8_t*)(f32_input ? m->tiles_f32[1].p : m->tiles_dev2.p)};
  auto issue_copy = [&](int64_t i0c, int slot) -> int {
    const int nbc = (int)((n - i0c < B) ? (n - i0c) : B);
    BQ_CUDA(ctx, cudaStreamWaitEvent(m->copy_stream, m->consumed[slot], 0));   // previous reader of this slot done
    if (compressed) {
      const int rcu = enc->upload(ctx, i0c / B, slot, m->copy_stream);
      if (rcu) return rcu;
    } else {
      BQ_CUDA(ctx, cudaMemcpyAsync(stage[slot], tiles + (size_t)i0c * tile_bytes, (size_t)nbc * tile_bytes,
                                   cudaMemcpyHostToDevice, m->copy_stream));
    }
    BQ_CUDA(ctx, cudaEventRecord(m->copied[slot], m->copy_stream));
    return BQ_OK;
  };
  if (!tiles_on_dev && n > 0) {
    int rc0 = issue_copy(0, 0);
    if (rc0) return rc0;
  }
  int64_t batch_idx = 0;
  for (int64_t i0 = 0; i0 < n; i0 += B, ++batch_idx) {
    const int nb = (int)((n - i0 < B) ? (n - i0) : B);
    int rc;
    const int slot = (int)(batch_idx & 1);
    if (tiles_on_dev) {
      m->tiles_src = tiles + (size_t)i0 * tile_bytes;
    } else {
      BQ_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, m->copied[slot], 0));
      m->tiles_src = stage[slot];
      if (compressed) {
        if ((rc = enc->decode_group(ctx, batch_idx, slot, (uint8_t*)m->tiles_dev.p))) return rc;
        BQ_CUDA(ctx, cudaEventRecord(m->consumed[slot], ctx->stream));        // the compressed slot is free once decoded
        m->tiles_src = (const uint8_t*)m->tiles_dev.p;
      }
    }
    const uint8_t* mdev = nullptr;       // masks of the head batch (device)
    if (masks) {
      if (masks_on_dev) mdev = masks + (size_t)head_start * mask_per_tile;
      else {
        BQ_CUDA(ctx, cudaMemcpyAsync((uint8_t*)m->masks_dev.p + (size_t)head_count * mask_per_tile,
                                     masks + (size_t)i0 * mask_per_tile, (size_t)nb * mask_per_tile,
                                     cudaMemcpyHostToDevice, ctx->stream));
        mdev = (const uint8_t*)m->masks_dev.p;
      }
    }
    if (m->norm_kind == BQ_NORM_REINHARD_FAST && !f32_input) {
      if ((rc = bq_stain_launch(ctx, m->tiles_src, nb, m->px, (const float*)m->norm_lut.p, (float*)m->norm_stats.p,
                                m->norm_means, m->norm_stds, (uint8_t*)m->tiles_norm.p)))
        return rc;
      m->tiles_src = (const uint8_t*)m->tiles_norm.p;
    }
    if ((rc = run_backbone_graphed(m, nb))) return rc;
    if (!tiles_on_dev) {
      if (!compressed) BQ_CUDA(ctx, cudaEventRecord(m->consumed[slot], ctx->stream));
      // The next micro-batch's copy is issued AFTER this one's backbone is queued: a copy from PAGEABLE memory blocks the
      // calling thread while the driver stages it, and that time must fall under queued GPU work (from pinned memory the
      // call returns at once and the order makes no difference).
      if (i0 + B < n && (rc = issue_copy(i0 + B, slot ^ 1))) return rc;
    }
    if (features && (rc = bq_from_device(ctx, features + (size_t)i0 * kFeatures, m->feat.p, (size_t)nb * kFeatures * 4)))
      return rc;
    const bool last = i0 + B >= n;
    {
      // hidden_0 now (per micro-batch); the dropout-bearing layers once enough tiles are queued to fill the SMs
      // (site 0 only: the per-sample feature masks of THIS micro-batch -- its global tile index and its slice of the masks)
      if ((rc = run_head(m, nb, T, seed, tile_index_base + (uint64_t)i0,
                         mdev ? mdev + (size_t)head_count * mask_per_tile : nullptr, head_count, 0)))
        return rc;
      head_count += nb;
      if (last || head_count + B > m->head_batch) {
        if ((rc = run_head(m, 0, T, seed, tile_index_base + (uint64_t)head_start, mdev, 0, head_count))) return rc;
        if (m->profiling) cudaEventRecord(m->ev[6], ctx->stream);
        if ((rc = bq_from_device(ctx, mean + (size_t)head_start * NC, m->out_mean.p, (size_t)head_count * NC * 4)) ||
            (rc = bq_from_device(ctx, std + (size_t)head_start * NC, m->out_std.p, (size_t)head_count * NC * 4)))
          return rc;
        head_start += head_count;
        head_count = 0;
      } else if (m->profiling) {
        cudaEventRecord(m->ev[6], ctx->stream);
      }
    }
    kprofile_collect(m);
    if (m->profiling) {
      BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      for (int s = 0; s < 6; ++s) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, m->ev[s], m->ev[s + 1]) == cudaSuccess) m->stage_ms[s] += ms;
      }
    }
  }
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (compressed) return enc->finish(ctx, nullptr);
  return BQ_OK;
}

int bq_model_debug_stage(bq_model* m, const uint8_t* tiles, int64_t n, const char* stage, float* out,
                         int64_t out_capacity, int64_t out_shape[4]) {
  if (!m) return BQ_ERR_ARG;
  bq_ctx* ctx = m->ctx;
  if (!m->weights_loaded) return bq_fail(ctx, BQ_ERR_STATE, "weights not loaded");
  if (!tiles || !stage || !out || !out_shape || n < 1 || n > m->max_batch)
    return bq_fail(ctx, BQ_ERR_ARG, "bq_model_debug_stage: bad argument (n must be <= max_batch)");
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc;
  if ((rc = stage_tiles(m, tiles, (int)n))) return rc;
  const std::string tag(stage);
  const Op* op = nullptr;
  const int prof = m->profiling;
  m->profiling = 0;
  rc = run_backbone(m, (int)n, &tag, &op);
  m->profiling = prof;
  if (rc) return rc;
  if (!op) return bq_fail(ctx, BQ_ERR_ARG, "unknown stage '%s'", stage);
  const bf16* src = op->kind == OP_GEMM ? op->gp.out : op->out;
  const int64_t h = op->Ho, w = op->kind == OP_CONV1 ? op->Ho : op->Wo, c = op->kind == OP_CONV1 ? 32 : op->Cout;
  const int64_t total = n * h * w * c;
  out_shape[0] = n; out_shape[1] = h; out_shape[2] = w; out_shape[3] = c;
  if (total > out_capacity) return bq_fail(ctx, BQ_ERR_ARG, "output buffer too small: need %lld floats", (long long)total);
  void* scr = nullptr;
  if ((rc = bq_scratch(ctx, total * 4, &scr))) return rc;
  if (op->padded_out) {
    // zero-padded 20 x 20 layout -> dense [n, 19, 19, 728] behind the fp32 area of the scratch buffer
    if ((rc = bq_scratch(ctx, total * 4 + total * 2 + 256, &scr))) return rc;
    bf16* dense = (bf16*)((char*)scr + ((total * 4 + 255) / 256) * 256);
    bq::sepmid::pad_copy_kernel<<<1024, 256, 0, ctx->stream>>>(src, dense, (int)n, 0);
    BQ_LAUNCH_CHECK(ctx);
    src = dense;
  }
  bf16_to_f32_kernel<<<1024, 256, 0, ctx->stream>>>(src, (float*)scr, total);
  BQ_LAUNCH_CHECK(ctx);
  if ((rc = bq_from_device(ctx, out, scr, total * 4))) return rc;
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BQ_OK;
}

int bq_model_debug_tags(bq_model* m, char* out, int64_t capacity) {
  if (!m) return BQ_ERR_ARG;
  std::string all;
  for (const Op& op : m->plan)
    if (!op.tag.empty()) all += op.tag + "\n";
  if (!out || (int64_t)all.size() + 1 > capacity)
    return bq_fail(m->ctx, BQ_ERR_ARG, "bq_model_debug_tags: need %lld bytes", (long long)all.size() + 1);
  memcpy(out, all.c_str(), all.size() + 1);
  return BQ_OK;
}

int bq_model_debug_h1(bq_model* m, int64_t n, float* out) {
  if (!m) return BQ_ERR_ARG;
  bq_ctx* ctx = m->ctx;
  if (!out || n < 1 || n > m->head_batch || !m->h_act[0].p || m->head_T < 1)
    return bq_fail(ctx, BQ_ERR_ARG, "bq_model_debug_h1: needs a preceding predict of >= n tiles (n <= %d)", m->head_batch);
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  // with dropout on the pooled features hidden_0 is per sample: [n * T, W] rows in (tile, sample) order
  const int64_t rows = (m->sites & 1) ? n * m->head_T : n;
  const int64_t total = rows * m->cfg.hidden_width;
  void* scr = nullptr;
  int rc;
  if ((rc = bq_scratch(ctx, total * 4, &scr))) return rc;
  bf16_to_f32_kernel<<<1024, 256, 0, ctx->stream>>>((const bf16*)m->h_act[0].p, (float*)scr, total);
  BQ_LAUNCH_CHECK(ctx);
  if ((rc = bq_from_device(ctx, out, scr, total * 4))) return rc;
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BQ_OK;
}

int bq_model_set_normalizer(bq_model* m, int32_t kind, const float target_means[3], const float target_stds[3]) {
  if (!m) return BQ_ERR_ARG;
  bq_ctx* ctx = m->ctx;
  if (kind == BQ_NORM_NONE) { m->norm_kind = BQ_NORM_NONE; return BQ_OK; }
  if (kind != BQ_NORM_REINHARD_FAST) return bq_fail(ctx, BQ_ERR_ARG, "bq_model_set_normalizer: unknown normaliser %d", kind);
  if (!target_means || !target_stds) return bq_fail(ctx, BQ_ERR_ARG, "bq_model_set_normalizer: null target statistics");
  for (int i = 0; i < 3; ++i) {
    if (!(target_stds[i] > 0.f)) return bq_fail(ctx, BQ_ERR_ARG, "bq_model_set_normalizer: target_stds must be > 0");
    m->norm_means[i] = target_means[i];
    m->norm_stds[i] = target_stds[i];
  }
  BQ_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc;
  if ((rc = bq_alloc(ctx, m->tiles_norm, (size_t)m->max_batch * m->px * m->px * 3)) ||
      (rc = bq_alloc(ctx, m->norm_stats, (size_t)m->max_batch * 6 * sizeof(float))) ||
      (rc = bq_alloc(ctx, m->norm_lut, 256 * sizeof(float))))
    return rc;
  float lut[256];
  bq::stain::build_gamma_lut(lut);
  BQ_CUDA(ctx, cudaMemcpyAsync(m->norm_lut.p, lut, sizeof(lut), cudaMemcpyHostToDevice, ctx->stream));
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  m->norm_kind = kind;
  return BQ_OK;
}

int bq_model_set_profiling(bq_model* m, int enabled) {
  if (!m) return BQ_ERR_ARG;
  m->profiling = enabled < 0 ? 0 : (enabled > 2 ? 2 : enabled);
  return BQ_OK;
}

int bq_model_kernel_profile(bq_model* m, double ms[BQ_PROFILE_KINDS], double flops[BQ_PROFILE_KINDS],
                            double bytes[BQ_PROFILE_KINDS], int64_t launches[BQ_PROFILE_KINDS]) {
  if (!m || !ms || !flops || !bytes || !launches) return BQ_ERR_ARG;
  for (int k = 0; k < BQ_PROFILE_KINDS; ++k) {
    ms[k] = m->k_ms[k]; flops[k] = m->k_flops[k]; bytes[k] = m->k_bytes[k]; launches[k] = m->k_launches[k];
  }
  return BQ_OK;
}

int bq_model_last_stage_ms(bq_model* m, float ms[8]) {
  if (!m || !ms) return BQ_ERR_ARG;
  for (int i = 0; i < 8; ++i) ms[i] = m->stage_ms[i];
  return BQ_OK;
}

}  // extern "C"
