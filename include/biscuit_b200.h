/*
 * biscuit_b200.h -- C ABI of libbiscuit_b200.so (hand-written sm_100a kernels for BISCUIT's hot path).
 *
 * The reference (jamesdolezal/biscuit) is pure Python and has no FFI of its own; its boundary for this
 * path is the Python call surface of biscuit/threshold.py and Slideflow's UncertaintyInterface.  This
 * header is the boundary a maintainer would bind underneath that surface (ctypes stub in INTEGRATION.md).
 * Each entry point cites the reference interface it replaces (file:line under the upstream repo).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (BQ_ERR_*); bq_last_error() gives the message.
 *     No C++ exception crosses the boundary.
 *   - the caller allocates every output; the library never frees caller memory.
 *   - data pointers may be HOST or DEVICE memory (resolved with cudaPointerGetAttributes); host buffers
 *     are staged through the context's stream, device buffers are used in place.
 *   - one bq_ctx per GPU and per host thread; a ctx is not thread-safe.
 *   - strings never cross the ABI: slide / patient names are factorised by the caller into int32
 *     first-appearance codes (code < 0 == missing key, skipped like pandas' dropna).
 */
#ifndef BISCUIT_B200_H
#define BISCUIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BQ_ABI_VERSION 1

enum {
  BQ_OK = 0,
  BQ_ERR_CUDA = -1,      /* CUDA runtime / driver failure                         */
  BQ_ERR_ARG = -2,       /* bad argument (null pointer, negative size, bad enum)  */
  BQ_ERR_STATE = -3,     /* call order violated (e.g. predict before weights)     */
  BQ_ERR_WEIGHTS = -4,   /* missing / mis-shaped weight tensor                    */
  BQ_ERR_NOMEM = -5,
  BQ_ERR_DATA = -6       /* malformed input data (a JPEG / PNG tile, a TFRecord)  */
};

enum { BQ_F32 = 0, BQ_F64 = 1 };

typedef struct bq_ctx bq_ctx;
typedef struct bq_table bq_table;
typedef struct bq_model bq_model;

/* ------------------------------------------------------------------------------------------------
 * context
 * ---------------------------------------------------------------------------------------------- */
int bq_abi_version(void);
int bq_create(int device, bq_ctx** out);
void bq_destroy(bq_ctx* ctx);
/* message of the last failing call on this ctx (ctx == NULL: last failing bq_create on this thread) */
const char* bq_last_error(bq_ctx* ctx);
/* number of kernels this library has launched on ctx since creation (bench.py's `gpu_launches`) */
int64_t bq_launch_count(bq_ctx* ctx);
int bq_sync(bq_ctx* ctx);
/* the cudaStream_t all work of this ctx is enqueued on (so callers can time it with CUDA events) */
void* bq_stream(bq_ctx* ctx);

/* ------------------------------------------------------------------------------------------------
 * tile-prediction tables  (replaces the pandas DataFrame plumbing of biscuit/threshold.py)
 * ---------------------------------------------------------------------------------------------- */

/* Upload / wrap one tile table: y_pred, uncertainty in `dtype`, y_true as uint8, n rows.
 * Columns are the ones biscuit/utils.py:31-53 (rename_cols) produces. */
int bq_table_create(bq_ctx* ctx, int64_t n, int dtype, const void* y_pred, const void* uncertainty,
                    const uint8_t* y_true, bq_table** out);
void bq_table_destroy(bq_table* t);

/* group keys for process_group_predictions (threshold.py:190-192): first-appearance codes of df[level] */
int bq_table_set_groups(bq_table* t, const int32_t* codes, int32_t n_groups);

/* input validation done by threshold.py:141 (NaN in y_pred) and by sklearn's roc_curve
 * (assert_all_finite, binary labels).  flags[0]=#NaN y_pred, [1]=#non-finite y_pred,
 * [2]=#non-finite uncertainty, [3]=#labels outside {0,1}. */
int bq_table_validate(bq_table* t, int64_t flags[4]);

/* threshold.py:170-176: error=|y_true-y_pred| (float64, as int64-float promotion gives), correct,
 * incorrect (kept on the device for bq_tile_roc), y_pred_bin = y_pred >= pred_thresh.
 * `pred_thresh` must already carry NumPy's scalar-promotion semantics (see INTEGRATION.md).
 * Any output pointer may be NULL. */
int bq_tile_process(bq_table* t, double pred_thresh, double* error, uint8_t* correct,
                    uint8_t* y_pred_bin);

typedef struct bq_roc_result {
  double threshold;   /* Youden-optimal threshold (+inf when the prepended (0,0) point wins)   */
  double youden_j;    /* max(tpr - fpr) in float64                                             */
  double auc;         /* sklearn.metrics.auc(fpr, tpr); NaN when a class is absent             */
  int64_t n_pos, n_neg;
  int64_t n_points;   /* ROC points after sklearn's drop_intermediate, incl. the (0,0) point    */
  int64_t best_index; /* index into that curve                                                 */
  int32_t status;     /* 0 ok; 1 single-class labels (reference idiom raises ValueError); 2 empty */
  int32_t auc_exact;  /* 1: AUC summed in numpy's pairwise order (bit-exact); 0: parallel sum    */
} bq_roc_result;

enum { BQ_SCORE_Y_PRED = 0, BQ_SCORE_UNCERTAINTY = 1 };
enum { BQ_LABEL_Y_TRUE = 0, BQ_LABEL_INCORRECT = 1 };

/* sklearn.metrics.roc_curve + the reference's Youden idiom over ALL rows of the table:
 * threshold.py:145-152 (y_true vs y_pred) and threshold.py:419-424 (incorrect vs uncertainty). */
int bq_tile_roc(bq_table* t, int score_sel, int label_sel, bq_roc_result* out);

/* same on caller arrays; `include` (nullable) restricts to rows with include[i] != 0.
 * threshold.py:212-220 (group ROC), 451-456 (slide UQ ROC), utils.py:487-504 (auc). */
int bq_roc(bq_ctx* ctx, const void* score, int dtype, const uint8_t* label, const uint8_t* include,
           int64_t n, bq_roc_result* out);

/* threshold.py:298 / 412 / 426: keep rows with uncertainty < tile_uq (compared in float64, the caller
 * rounds tile_uq to float32 first when NumPy would).  enabled == 0 removes the filter. */
int bq_table_set_tile_filter(bq_table* t, int enabled, double tile_uq);

/* threshold.py:191-204: per-group mean of y_pred / uncertainty (row-order Kahan sum in the column
 * dtype, as pandas group_mean), mean of y_true (float64), surviving row count and first surviving row
 * (for first-appearance ordering, -1 when the group lost all rows).  Arrays have n_groups entries. */
int bq_group_reduce(bq_table* t, void* g_pred, void* g_unc, double* g_true_mean, int64_t* g_count,
                    int64_t* g_first_row);

enum { BQ_KEEP_ALL = 0, BQ_KEEP_HIGH_CONFIDENCE = 1, BQ_KEEP_LOW_CONFIDENCE = 2 };

/* threshold.py:228-244 (error / correct / incorrect / y_pred_bin per group, `>= pred_thresh`),
 * 323-330 (include = unc < slide_uq, or >= for low confidence) and 339-345 (confusion counts among the
 * included groups with the STRICT `y_pred > slide_pred`).  confusion = {tp, fp, tn, fn}. */
int bq_group_apply(bq_ctx* ctx, int64_t n_groups, int dtype, const void* g_pred, const void* g_unc,
                   const uint8_t* g_true, double pred_thresh, double slide_pred_strict, int keep_mode,
                   double slide_uq, void* error, uint8_t* correct, uint8_t* incorrect,
                   uint8_t* y_pred_bin, uint8_t* include, int64_t confusion[4]);

/* ------------------------------------------------------------------------------------------------
 * Xception-UQ Monte-Carlo-dropout inference
 * (replaces slideflow.model.tensorflow.UncertaintyInterface.__call__, call site results.py:234,257;
 *  architecture contract biscuit/hp.py:3-24)
 * ---------------------------------------------------------------------------------------------- */

typedef struct bq_model_config {
  int32_t tile_px;        /* 299  (hp.py:5)                    */
  int32_t hidden_width;   /* 1024 (hp.py:13); a multiple of 64, at most 1024 (the fused head's limit) */
  int32_t hidden_layers;  /* 2    (hp.py:21)                   */
  int32_t n_classes;      /* 2; 2..8                           */
  float dropout;          /* 0.1  (hp.py:11)                   */
  int32_t max_batch;      /* tiles per backbone micro-batch    */
  /* MC-dropout placement, bit i = a Dropout(rate) active at inference after site i:
   *   bit 0: the pooled 2048-d features (Slideflow's `post_convolution`), bit 1: hidden_0, bit 2: hidden_1.
   * 0 selects the default 0b110 (after each hidden layer), so a model without any dropout site cannot be built: the
   * Python `ModelConfig` rejects an all-False placement instead of passing 0.  Which placement a saved model has
   * depends on the Slideflow version that built it (hp.py:11-12 only fix the rate and `uq`); INTEGRATION.md lists both. */
  int32_t dropout_sites;
  int32_t reserved[7];
} bq_model_config;

typedef struct bq_named_tensor {
  const char* name;       /* Keras layer/variable name, e.g. "block2_sepconv1/depthwise_kernel" */
  const float* data;      /* host fp32, Keras layout (HWIO conv kernels, [in,out] dense)         */
  int32_t ndim;
  int64_t shape[4];
} bq_named_tensor;

int bq_model_create(bq_ctx* ctx, const bq_model_config* cfg, bq_model** out);
void bq_model_destroy(bq_model* m);
/* folds BatchNorm (eps 1e-3) into per-channel scale/shift, pads 728->736 channels, converts to bf16 */
int bq_model_load_weights(bq_model* m, const bq_named_tensor* tensors, int32_t n_tensors);

/* One call = standardise + backbone (once) + T dropout-head samples + mean/std (population, ddof=0).
 *   tiles   uint8 NHWC [n, px, px, 3] (host or device)
 *   T       MC-dropout samples (Slideflow: 30)
 *   seed, tile_index_base   Philox key / first global tile index (so shards draw disjoint streams)
 *   masks   nullable injected keep-masks uint8 [n, T, hidden_layers, hidden_width] (1 = keep)
 *   mean, std   float32 [n, n_classes]   (y_pred / uncertainty columns of utils.py:19-28 = class 1)
 *   features    nullable float32 [n, 2048] post-pooling features                                   */
/* injected keep-masks (parity tests): uint8 [n, T, n_enabled_sites, mask_width], enabled sites in ascending order,
 * mask_width = 2048 when site 0 is enabled, else hidden_width */
int bq_predict_uq(bq_model* m, const uint8_t* tiles, int64_t n, int32_t T, uint64_t seed,
                  uint64_t tile_index_base, const uint8_t* masks, float* mean, float* std,
                  float* features);

/* The reference's LITERAL call (results.py:255-257): tiles already passed through tf.image.per_image_standardization,
 * float32 NHWC [n, 299, 299, 3].  Same outputs; the tile statistics, the standardisation and the stain normaliser are
 * skipped (the first convolution reads the floats as they are). */
int bq_predict_uq_standardized(bq_model* m, const float* tiles, int64_t n, int32_t T, uint64_t seed,
                               uint64_t tile_index_base, const uint8_t* masks, float* mean, float* std, float* features);

/* Debug / parity hooks: run only the backbone, returning bf16-rounded activations of a named stage as
 * float32 (NHWC).  Used by tests to localise a mismatch; not part of the reference surface. */
int bq_model_debug_stage(bq_model* m, const uint8_t* tiles, int64_t n, const char* stage, float* out,
                         int64_t out_capacity, int64_t out_shape[4]);
/* hidden_0 activations (bf16 as float32) of the first n tiles of the last bq_predict_uq call, when that call held them
 * in one head batch: [n, hidden_width], or [n, T, hidden_width] (one row per sample, T of that call) when dropout on
 * the pooled features is on.  `out` must hold that many floats. */
int bq_model_debug_h1(bq_model* m, int64_t n, float* out);
/* the debug_stage tags of the execution plan in execution order, one per line (NUL-terminated) */
int bq_model_debug_tags(bq_model* m, char* out, int64_t capacity);

/* per-stage device time of the last bq_predict_uq call, in ms: {stats+conv1, conv2, entry, middle,
 * exit, head} -- measured with CUDA events on the ctx stream when enabled */
int bq_model_set_profiling(bq_model* m, int enabled);   /* 0 off, 1 per stage, 2 per kernel family */
int bq_model_last_stage_ms(bq_model* m, float ms[8]);

/* Per-kernel-family accounting of the last bq_predict_uq call (profiling level 2): summed CUDA-event time
 * of every launch of the family on the ctx stream, the ALGORITHMIC flops / bytes those launches processed
 * (DESIGN.md states the per-unit figures) and the launch count.  bench.py's `roofline` is built from this. */
enum {
  BQ_K_STATS = 0, BQ_K_CONV1 = 1, BQ_K_GEMM_CONV2 = 2, BQ_K_GEMM_PW = 3, BQ_K_DW = 4, BQ_K_POOLADD = 5,
  BQ_K_SUBSAMPLE = 6, BQ_K_GAP = 7, BQ_K_HEAD_GEMM = 8, BQ_K_MC_EXPAND = 9, BQ_K_HEAD_FINAL = 10,
  BQ_K_HEAD_FUSED = 11, BQ_K_SEP_FUSED = 12, BQ_K_SEP_MID = 13,
  BQ_PROFILE_KINDS = 16
};
int bq_model_kernel_profile(bq_model* m, double ms[BQ_PROFILE_KINDS], double flops[BQ_PROFILE_KINDS],
                            double bytes[BQ_PROFILE_KINDS], int64_t launches[BQ_PROFILE_KINDS]);

/* ------------------------------------------------------------------------------------------------
 * slide tile-grid heat map with uncertainty masking
 *   replaces the array side of `hm = sf.Heatmap(slide, model)` + `hm.uncertainty[:, :, 0] > thresh` +
 *   `hm.logits[uq_mask, :] = [-1, -1]` (results.py:216-227); tile extraction and rendering are Slideflow's.
 * ---------------------------------------------------------------------------------------------- */
/* logits / uncertainty [gy, gx, n_classes] float32: -1 everywhere, then cell (x, y) = grid_xy[t] of tile t receives
 * mean[t] / stdv[t] (outputs of bq_predict_uq). */
int bq_heatmap_build(bq_ctx* ctx, int64_t n, int32_t n_classes, const float* mean, const float* stdv, const int32_t* grid_xy,
                     int32_t gx, int32_t gy, float* logits, float* uncertainty);
/* mask[cell] = uncertainty[cell][0] > thresh (float64 compare; apply NumPy's scalar promotion to `thresh` first);
 * logits of masked cells := -1 in place. */
int bq_heatmap_mask(bq_ctx* ctx, int64_t cells, int32_t n_classes, const float* uncertainty, double thresh, float* logits,
                    uint8_t* mask);

/* ------------------------------------------------------------------------------------------------
 * multi-GPU exchange (one process -- or host thread -- per GPU; SURVEY.md 8e)
 *   The reference is single-process (no collective anywhere under /root/reference).  Here tiles shard over GPUs by whole
 *   slides, so the per-slide reduction (threshold.py:191-192) stays local and bit-exact; what crosses GPUs is
 *     - the per-slide aggregates {code, count, first_row, y_pred, uncertainty, y_true_mean} (6 x float64 per slide)
 *       before the slide-level stage of `apply` (threshold.py:304-348) / `detect` (threshold.py:433-468), and
 *     - for `detect` only, the per-tile (y_pred, uncertainty, y_true) triples feeding the cohort-wide tile ROCs
 *       (threshold.py:145-152, 419-424).
 *   Both are all-gathers of one byte block per rank.
 * ---------------------------------------------------------------------------------------------- */
#define BQ_COMM_ID_BYTES 128
/* rank 0 creates the NCCL unique id and hands it to the other ranks by any host-side means (file, MPI, pipe ...) */
int bq_comm_unique_id(uint8_t id[BQ_COMM_ID_BYTES]);
/* collective over all ranks: attaches an NCCL communicator (NVLink / NVSwitch) to this context */
int bq_comm_init(bq_ctx* ctx, int32_t rank, int32_t world, const uint8_t id[BQ_COMM_ID_BYTES]);
int bq_comm_size(bq_ctx* ctx, int32_t* rank, int32_t* world);   /* (0, 1) without a communicator */
void bq_comm_destroy(bq_ctx* ctx);
/* every rank sends `nbytes` (the same on all ranks; callers pad to the largest block) and receives world * nbytes in
 * rank order.  Host or device pointers; runs on the ctx stream and returns when `recv` is complete. */
int bq_allgather_bytes(bq_ctx* ctx, const void* send, int64_t nbytes, void* recv);

/* ------------------------------------------------------------------------------------------------
 * stain normalisation in front of per-image standardisation
 *   replaces `interface.wsi_normalizer.rgb_to_rgb(image)` (results.py:251-254) for hp.normalizer ==
 *   'reinhard_fast' (biscuit/hp.py:19); arithmetic restated from slideflow/norm/tensorflow/reinhard.py
 * ---------------------------------------------------------------------------------------------- */
enum { BQ_NORM_NONE = 0, BQ_NORM_REINHARD_FAST = 1 };
/* tiles, out: uint8 NHWC [n, px, px, 3] (host or device); target_means / target_stds: the fitted LAB
 * statistics of the reference image (3 floats each, host); lab_stats: nullable float32 [n, 6] =
 * per-tile {mean L, a, b, std L, a, b} of the SOURCE tiles (host or device). */
int bq_stain_normalize(bq_ctx* ctx, int32_t kind, const uint8_t* tiles, int64_t n, int32_t px,
                       const float target_means[3], const float target_stds[3], uint8_t* out,
                       float* lab_stats);
/* Make bq_predict_uq normalise every tile first (kind = BQ_NORM_NONE switches it off again). */
int bq_model_set_normalizer(bq_model* m, int32_t kind, const float target_means[3], const float target_stds[3]);

/* ------------------------------------------------------------------------------------------------
 * compressed tiles: baseline JPEG decode on the GPU and TFRecord reading
 *   replaces the host side of Slideflow's evaluate route (TFRecord read + per-tile JPEG decode in front of
 *   interface(batch)).  Decoded pixels equal libjpeg-turbo's default decompression byte for byte (JDCT_ISLOW,
 *   fancy upsampling, jdcolor.c YCbCr->RGB), i.e. PIL.Image.open(...).convert("RGB").
 *   Tiles are n JPEG files back to back: tile i = data[offsets[i], offsets[i + 1]); offsets is always host memory.
 *   Accepted: SOF0 / SOF1 8-bit Huffman, one interleaved scan of 3 components (YCbCr), sampling 4:4:4, 4:2:2 or 4:2:0,
 *   any DQT / DHT, restart intervals, APPn / COM segments (skipped), size px x px.
 * ---------------------------------------------------------------------------------------------- */
enum {
  BQ_JPEG_OK = 0,
  BQ_JPEG_NOT_JPEG = 1,            /* no SOI marker                                                  */
  BQ_JPEG_TRUNCATED_HEADER = 2,    /* the file ends inside its headers                               */
  BQ_JPEG_PROGRESSIVE = 3,
  BQ_JPEG_ARITHMETIC = 4,
  BQ_JPEG_LOSSLESS = 5,            /* lossless or hierarchical                                        */
  BQ_JPEG_PRECISION = 6,           /* not 8-bit samples                                               */
  BQ_JPEG_GRAYSCALE = 7,           /* 1 component                                                     */
  BQ_JPEG_CMYK = 8,                /* 4 components                                                    */
  BQ_JPEG_COMPONENTS = 9,          /* any other component count                                       */
  BQ_JPEG_SIZE = 10,               /* width or height differs from px                                 */
  BQ_JPEG_SAMPLING = 11,           /* sampling factors other than 4:4:4 / 4:2:2 / 4:2:0               */
  BQ_JPEG_MISSING_DQT = 12,
  BQ_JPEG_MISSING_DHT = 13,
  BQ_JPEG_BAD_TABLE = 14,          /* malformed DQT / DHT                                             */
  BQ_JPEG_BAD_HEADER = 15,         /* missing SOF / SOS / EOI, unexpected marker, bad scan parameters */
  BQ_JPEG_COLORSPACE = 16,         /* 3 components that are not YCbCr (Adobe transform 0, RGB ids)    */
  /* found on the device while decoding the entropy-coded segment */
  BQ_JPEG_BAD_ENTROPY_MARKER = 20, /* a marker other than RSTn inside the scan, or wrong RSTn sequence  */
  BQ_JPEG_INVALID_CODE = 21,       /* a Huffman code that is in no table                               */
  BQ_JPEG_TRUNCATED_DATA = 22      /* the scan ends before its last MCU                                */
};
/* one line of text per status code above */
const char* bq_jpeg_status_string(int32_t status);
/* Host only, no device needed: the marker parse bq_jpeg_decode runs first.  status[i] = BQ_JPEG_* of tile i.
 * data must be host memory.  Returns BQ_OK also when some tiles are rejected. */
int bq_jpeg_inspect(const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, int32_t* status);
/* Decode n tiles into out_u8 = uint8 NHWC [n, px, px, 3] (host or device); data host or device (device bytes are read
 * in place).  status[i] (host, nullable) = BQ_JPEG_* of tile i.  A rejected header fails the call with BQ_ERR_DATA
 * before anything is launched; an entropy-coded segment that runs out of bits or holds an invalid code fails it with
 * BQ_ERR_DATA after the batch (the other tiles are decoded; the rejected tile's pixels are 0). */
int bq_jpeg_decode(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, uint8_t* out_u8,
                   int32_t* status);
/* Subsequence statistics of the last bq_jpeg_decode on ctx, summed over its tiles: {tiles, subsequences,
 * synchronisation rounds (max over tiles), subsequences decoded again}. */
int bq_jpeg_last_stats(bq_ctx* ctx, int64_t stats[4]);
/* bq_predict_uq on JPEG tiles: same outputs, seeds and tile indices as bq_predict_uq on the decoded uint8 tiles.  The
 * compressed bytes of micro-batch i + 1 are copied while micro-batch i runs; each is decoded on the GPU into the
 * micro-batch buffer the uint8 path stages into. */
int bq_predict_uq_jpeg(bq_model* m, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t T, uint64_t seed,
                       uint64_t tile_index_base, const uint8_t* masks, float* mean, float* std, float* features);

/* PNG tiles, decoded on the GPU: the pixels equal PIL.Image.open(...).convert("RGB") (PNG is lossless, so also
 * TensorFlow's decode_png).  Same layout as the JPEG entry points: tile i = data[offsets[i], offsets[i + 1]), offsets
 * in host memory.  Accepted: 8-bit RGB (colour type 2), non-interlaced, px x px, any zlib level / strategy / window,
 * IDAT split into chunks of any size, ancillary chunks and PLTE (skipped).  Every chunk before the first IDAT must pass
 * its CRC; IDAT CRCs are not checked (the zlib Adler-32 is). */
enum {
  BQ_PNG_OK = 0,
  BQ_PNG_NOT_PNG = 1,              /* no PNG signature                                                */
  BQ_PNG_TRUNCATED_HEADER = 2,     /* the file ends before the first IDAT and the zlib header          */
  BQ_PNG_BAD_CRC = 3,              /* a chunk before the first IDAT fails its CRC                       */
  BQ_PNG_BAD_IHDR = 4,             /* IHDR missing / not first / length != 13 / invalid field / twice   */
  BQ_PNG_SIZE = 5,                 /* width or height differs from px                                  */
  BQ_PNG_BIT_DEPTH = 6,            /* not 8 bits per sample                                            */
  BQ_PNG_COLOUR_TYPE = 7,          /* grayscale, palette or alpha                                      */
  BQ_PNG_INTERLACED = 8,           /* Adam7                                                            */
  BQ_PNG_UNKNOWN_CRITICAL = 9,     /* a critical chunk other than IHDR / PLTE / IDAT / IEND            */
  BQ_PNG_NO_IDAT = 10,             /* IEND before any IDAT                                             */
  BQ_PNG_BAD_ZLIB = 11,            /* zlib header: CM != 8, CINFO > 7 or bad FCHECK                    */
  BQ_PNG_PRESET_DICT = 12,         /* zlib FDICT set                                                   */
  /* found on the device */
  BQ_PNG_TRUNCATED_DATA = 20,      /* the IDAT run or the DEFLATE stream ends early, or no Adler-32    */
  BQ_PNG_BAD_BLOCK = 21,           /* BTYPE 3, or a stored block with LEN != ~NLEN                     */
  BQ_PNG_BAD_HUFFMAN = 22,         /* over-subscribed / incomplete code, bad repeat, invalid symbol    */
  BQ_PNG_BAD_DISTANCE = 23,        /* a match reaching before the start of the stream                  */
  BQ_PNG_WRONG_SIZE = 24,          /* decompressed size != px * (1 + 3 px)                             */
  BQ_PNG_ADLER = 25,               /* Adler-32 mismatch                                                */
  BQ_PNG_BAD_FILTER = 26           /* a row filter type > 4                                            */
};
/* one line of text per status code above */
const char* bq_png_status_string(int32_t status);
/* Host only, no device needed: the chunk parse bq_png_decode runs first.  status[i] = BQ_PNG_* of tile i.  data must
 * be host memory.  Returns BQ_OK also when some tiles are rejected. */
int bq_png_inspect(const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, int32_t* status);
/* Decode n tiles into out_u8 = uint8 NHWC [n, px, px, 3] (host or device); data host or device (device bytes are read
 * in place).  status[i] (host, nullable) = BQ_PNG_* of tile i.  A rejected header fails the call with BQ_ERR_DATA
 * before anything is launched; a tile rejected on the device fails it with BQ_ERR_DATA after the batch (the other
 * tiles are decoded).  Stricter than Pillow on corrupt data: a missing Adler-32 and a stream that decompresses to
 * more bytes than the image are rejected. */
int bq_png_decode(bq_ctx* ctx, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t px, uint8_t* out_u8,
                  int32_t* status);
/* bq_predict_uq on PNG tiles: same outputs, seeds and tile indices as bq_predict_uq on the decoded uint8 tiles. */
int bq_predict_uq_png(bq_model* m, const uint8_t* data, const int64_t* offsets, int64_t n, int32_t T, uint64_t seed,
                      uint64_t tile_index_base, const uint8_t* masks, float* mean, float* std, float* features);

/* TFRecord file (uncompressed) in a host buffer: record framing {u64 length, masked CRC32C of the length, payload,
 * masked CRC32C of the payload}, both CRCs verified (SSE4.2 crc32 when the CPU has it), payload parsed as a
 * tf.train.Example.  For each record r < capacity: image[2r..2r+1] = byte range [begin, end) of the first value of the
 * bytes feature `image_key`, slide[2r..] = same for `slide_key` (-1, -1 when absent), loc[2r], loc[2r + 1] = first value
 * of the int64 features `x_key`, `y_key` (INT64_MIN when absent).  *n_records = records in the buffer (may exceed
 * capacity: call again with more room).  A bad CRC, a truncated record, a malformed Example, a record without
 * `image_key` or a gzip / zlib-compressed file fail with BQ_ERR_DATA and a message in err (err_capacity bytes). */
int bq_tfrecord_scan(const uint8_t* buf, int64_t len, const char* image_key, const char* slide_key, const char* x_key,
                     const char* y_key, int64_t capacity, int64_t* n_records, int64_t* image, int64_t* slide,
                     int64_t* loc, char* err, int64_t err_capacity);
/* CRC32C (Castagnoli) of a host buffer, and TFRecord's masked form ((crc >> 15 | crc << 17) + 0xa282ead8) */
uint32_t bq_crc32c(const uint8_t* buf, int64_t len);
uint32_t bq_crc32c_masked(const uint8_t* buf, int64_t len);

/* ------------------------------------------------------------------------------------------------
 * evaluation metrics next to the path
 *   replaces the bootstrap loop of utils.prediction_metrics (biscuit/utils.py:428-440) and the midrank
 *   passes of delong.fastDeLong (biscuit/delong.py:60-69); the order-sensitive floating-point finish
 *   (np.cov, statistics.mean / variance, scipy.stats.norm) stays in the Python wrapper
 * ---------------------------------------------------------------------------------------------- */
/* counts[b] = {tp, fp, tn, fn} of the n_samp rows idx[b][0..n_samp) (uint8 y_true / thresholded y_pred, length n) */
int bq_bootstrap_confusion(bq_ctx* ctx, const uint8_t* y_true, const uint8_t* y_pred_bin, int64_t n,
                           const int64_t* idx, int32_t n_boot, int32_t n_samp, int64_t* counts);
/* v[i] = V01 placement value of a positive / V10 of a negative example (original order, float64);
 * tz_pos_sum = sum of the positives' midranks among all examples; n_pos = number of positives.  n <= 2^20. */
int bq_delong_placements(bq_ctx* ctx, const void* score, int32_t dtype, const uint8_t* label, int64_t n,
                         double* v, double* tz_pos_sum, int64_t* n_pos);

/* Developer hook (hardware probe, not on the product path): one 128x16x16 tcgen05.mma whose A operand starts `shift`
 * rows into a 128B-swizzled [rows x 64] bf16 tile, channel group cg, against an identity B in the no-swizzle layout;
 * base_offset_mode 1 sets the descriptor base_offset field to (addr >> 7) & 7.  out = float [128][16]. */
int bq_debug_umma_probe(bq_ctx* ctx, int rows, int shift, int cg, int base_offset_mode, const uint16_t* x_bf16,
                        float* out);

#ifdef __cplusplus
}
#endif
#endif /* BISCUIT_B200_H */
