"""Predict-with-uncertainty on the GPU -- drop-in for the Slideflow call BISCUIT makes:

    interface = sf.model.tensorflow.UncertaintyInterface(model)      # reference results.py:234
    logits, uncertainty = interface(batch)                            # reference results.py:257

`UncertaintyInterface(weights)(tiles)` returns ``(mean softmax [B, C], std [B, 1])`` exactly like
the reference call site consumes it (`uncertainty[0][0]`, results.py:258).  Differences that are
the point of the rewrite: the input is the RAW uint8 tile (decode + `per_image_standardization`,
results.py:255, are fused into the first convolution), the backbone runs once per tile instead of
T = 30 times, and the T dropout samples of the head are evaluated on the pooled features.

`predict_table` produces the tile-prediction table BISCUIT reads back from Slideflow
(columns per reference biscuit/utils.py:19-28: '{outcome}-y_pred1', '{outcome}-uncertainty1',
'{outcome}-y_true0'), ready for `biscuit_b200.threshold`.

All compute is in libbiscuit_b200.so (csrc/model.cu, gemm_sm100.cuh, layers.cuh).  No CPU path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import pandas as pd

from . import _ffi
from .hp import ModelConfig, nature2022
from .encoded import EncodedBatch, entry_point
from .utils import uncertainty_header, y_pred_header, y_true_header

FEATURES = 2048


def _as_named_tensors(weights: dict):
    keep = []          # keep numpy buffers alive for the duration of the call
    arr = (_ffi.NamedTensor * len(weights))()
    for i, (name, w) in enumerate(weights.items()):
        a = np.ascontiguousarray(w, dtype=np.float32)
        keep.append(a)
        arr[i].name = name.encode()
        arr[i].data = a.ctypes.data_as(C.c_void_p)
        arr[i].ndim = a.ndim
        for d in range(a.ndim):
            arr[i].shape[d] = a.shape[d]
    return arr, keep


# Micro-batch the benchmark runs at (the library's cap is 512).  The dominant kernel -- the fused middle-flow sepconv --
# splits a micro-batch of B tiles into ceil(400 B / 160) work items for 74 CTA pairs: B = 503 gives 1258 items = exactly
# 17 per pair, B = 512 gives 1280 = 17.3 (an 18th round with 22 of 74 pairs busy).  Measured: +0.9 % tiles/s (DESIGN.md 6).
BENCH_MICRO_BATCH = 503


class UncertaintyInterface:
    """MC-dropout Xception-UQ inference (Slideflow `UncertaintyInterface` call surface).

    Args:
        weights: dict name -> float32 array under Keras variable names
            ('block1_conv1/kernel', 'block2_sepconv1/depthwise_kernel', '..._bn/gamma', 'hidden_0/kernel',
            'prelogits/bias', ...; residual 1x1 convs are 'block{2,3,4,13}_res').
        config: `ModelConfig` (default `hp.nature2022`).
        max_batch: tiles per backbone micro-batch held on the device.
        device: CUDA device index (default LOCAL_RANK or 0).
        normalizer: None, 'reinhard_fast' (the reference's `hp.normalizer`, hp.py:19) or a
            `norm.ReinhardFastNormalizer` carrying the fit; tiles are then stain-normalised on the GPU
            in front of the per-image standardisation inside `predict`.
    """

    def __init__(self, weights: dict, config: ModelConfig = nature2022, max_batch: int = 64,
                 device: int | None = None, ctx: _ffi.Context | None = None, normalizer=None):
        if config.model != "xception" or config.pooling != "avg" or config.include_top:
            raise ValueError("only the reference configuration (xception, avg pooling, include_top=False) is built")
        if not config.uq:
            raise ValueError("UncertaintyInterface runs MC-dropout inference: config.uq must be True")
        self.config = config
        self.ctx = ctx or _ffi.default_context(device)
        self.lib = self.ctx.lib
        self.num_uq = config.uq_samples
        self.max_batch = int(max_batch)
        self._head_T = None
        self.wsi_normalizer = None     # attribute the reference call site probes (results.py:251)
        cfg = _ffi.ModelConfig(tile_px=config.tile_px, hidden_width=config.hidden_layer_width,
                               hidden_layers=config.hidden_layers, n_classes=config.n_classes,
                               dropout=config.dropout, max_batch=max_batch,
                               dropout_sites=config.dropout_site_mask)
        h = C.c_void_p()
        _ffi.check(self.ctx.handle, self.lib.bq_model_create(self.ctx.handle, C.byref(cfg), C.byref(h)),
                   "bq_model_create")
        self.h = h
        arr, keep = _as_named_tensors(weights)
        _ffi.check(self.ctx.handle, self.lib.bq_model_load_weights(self.h, arr, len(weights)),
                   "bq_model_load_weights")
        del keep
        if normalizer is not None:
            self.set_normalizer(normalizer)

    def set_normalizer(self, normalizer):
        """Stain normalisation applied to every tile inside `predict` (None switches it off).  The
        reference applies `interface.wsi_normalizer.rgb_to_rgb` itself before calling the interface
        (results.py:251-254); callers that keep doing so must leave this unset."""
        from . import norm
        if isinstance(normalizer, str):
            normalizer = norm.autoselect(normalizer)
        if normalizer is None:
            _ffi.check(self.ctx.handle, self.lib.bq_model_set_normalizer(self.h, norm.NORM_NONE, None, None),
                       "bq_model_set_normalizer")
        else:
            tm = np.ascontiguousarray(normalizer.target_means, np.float32)
            ts = np.ascontiguousarray(normalizer.target_stds, np.float32)
            _ffi.check(self.ctx.handle,
                       self.lib.bq_model_set_normalizer(self.h, int(normalizer.kind), _ffi.ptr(tm), _ffi.ptr(ts)),
                       "bq_model_set_normalizer")
        self.normalizer = normalizer

    def close(self):
        if getattr(self, "h", None):
            self.lib.bq_model_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------
    def predict(self, tiles, T: int | None = None, seed: int = 0, tile_index_base: int = 0,
                masks=None, return_features: bool = False, out_mean=None, out_std=None):
        """tiles: NHWC [n, 299, 299, 3] -- uint8 raw RGB (decode + per-image standardisation fused into the first
        convolution), or float32 ALREADY passed through `tf.image.per_image_standardization` as the reference's call site
        does (results.py:255-257); numpy, or a CUDA torch tensor used in place.  Or a `jpeg.JpegBatch` / `png.PngBatch`
        of JPEG / PNG tiles, decoded on the GPU in front of the backbone (a JpegBatch with its `dct_method` /
        `fancy_upscaling`, a PngBatch with its `convert_rgb`): the results equal `predict` on the decoded uint8 tiles bit for bit.
        Returns (mean [n, C], std [n, C]) float32 -- population std over T dropout samples."""
        T = int(T or self.num_uq)
        encoded = tiles.FORMAT if isinstance(tiles, EncodedBatch) else None
        n = len(tiles) if encoded else int(tiles.shape[0])
        px = self.config.tile_px
        if not encoded and tuple(tiles.shape[1:]) != (px, px, 3):
            raise ValueError(f"tiles must be [n, {px}, {px}, 3], got {tuple(tiles.shape)}")
        dt = encoded or str(tiles.dtype).replace("torch.", "")
        if dt not in ("uint8", "float32", "jpeg", "png"):
            raise TypeError("tiles must be uint8 (raw RGB) or float32 (already per-image standardised), got " + dt)
        if isinstance(tiles, np.ndarray):
            tiles = np.ascontiguousarray(tiles)
        elif hasattr(tiles, "is_contiguous") and not tiles.is_contiguous():
            raise ValueError("tiles must be contiguous (NHWC)")
        nc = self.config.n_classes
        mean = out_mean if out_mean is not None else np.empty((n, nc), np.float32)
        std = out_std if out_std is not None else np.empty((n, nc), np.float32)
        for name, buf in (("out_mean", mean), ("out_std", std)):    # raw pointers cross the ABI: check them here
            if not isinstance(buf, np.ndarray) or buf.dtype != np.float32 or buf.shape != (n, nc) or not buf.flags.c_contiguous:
                raise ValueError(f"{name} must be a C-contiguous float32 array of shape {(n, nc)}")
        feats = np.empty((n, FEATURES), np.float32) if return_features else None
        if masks is not None:
            sites = self.config.dropout_sites
            width = FEATURES if sites[0] else self.config.hidden_layer_width
            want = (n, T, sum(bool(x) for x in sites), width)
            if tuple(masks.shape) != want:
                raise ValueError(f"masks must have shape {want}")
            if isinstance(masks, np.ndarray):
                masks = np.ascontiguousarray(masks, dtype=np.uint8)
        if encoded:
            name, flags = entry_point(f"bq_predict_uq_{encoded}", tiles)
            rc = getattr(self.lib, name)(self.h, _ffi.ptr(tiles.data), _ffi.ptr(tiles.offsets), n, *flags, T,
                                         C.c_uint64(seed), C.c_uint64(tile_index_base), _ffi.ptr(masks), _ffi.ptr(mean),
                                         _ffi.ptr(std), _ffi.ptr(feats))
        else:
            entry = self.lib.bq_predict_uq if dt == "uint8" else self.lib.bq_predict_uq_standardized
            rc = entry(self.h, _ffi.ptr(tiles), n, T, C.c_uint64(seed), C.c_uint64(tile_index_base), _ffi.ptr(masks),
                       _ffi.ptr(mean), _ffi.ptr(std), _ffi.ptr(feats))
        _ffi.check(self.ctx.handle, rc, "bq_predict_uq")
        if n > 0:
            self._head_T = T             # the head buffers now hold this call's T (debug_h1)
        if return_features:
            return mean, std, feats
        return mean, std

    def __call__(self, tiles, **kw):
        """`logits, uncertainty = interface(batch)` (results.py:257): mean softmax [B, C] and the per-class std
        [B, C] over the dropout samples, so the reference's `uncertainty[0][0]` (results.py:258) reads the class-0 std --
        for two classes both stds agree up to rounding.  `batch` may be the standardised float32 batch the reference
        passes, raw uint8 tiles, a `jpeg.JpegBatch` or a `png.PngBatch`."""
        return self.predict(tiles, **kw)

    # ------------------------------------------------------------------------------------
    def debug_stage(self, tiles: np.ndarray, stage: str) -> np.ndarray:
        """Parity hook: NHWC float32 copy of the output of one op of the backbone plan, run up to that op.
        Tags: 'block1_conv1', 'block1_conv2'; 'block{b}_sub' (stride-2 subsample) and 'block{b}_res' (1x1 residual GEMM)
        for b in 2, 3, 4, 13; 'block{b}_sepconv{i}_dw' (a depthwise output, where the depthwise runs as its own kernel);
        'block{b}_sepconv{i}' (a SeparableConv after BatchNorm and ReLU); 'block{b}' for a block output: blocks 2-4 and 13
        after max-pool + residual, blocks 5-12 after the third sepconv + residual (no separate 'block{b}_sepconv3' tag),
        and 'block14' = block14_sepconv2 (no separate tag)."""
        n = int(tiles.shape[0])
        cap = n * 149 * 149 * 128
        out = np.empty(cap, np.float32)
        shape = (C.c_int64 * 4)()
        tiles = np.ascontiguousarray(tiles, dtype=np.uint8)
        _ffi.check(self.ctx.handle,
                   self.lib.bq_model_debug_stage(self.h, _ffi.ptr(tiles), n, stage.encode(), _ffi.ptr(out), cap, shape),
                   "bq_model_debug_stage")
        s = tuple(int(x) for x in shape)
        return out[: int(np.prod(s))].reshape(s).copy()

    def debug_h1(self, n: int) -> np.ndarray:
        """Parity hook: hidden_0 output (bf16 as float32) of the first n tiles of the last `predict` call, which must
        have held them in one head batch: [n, hidden_width], or [n, T, hidden_width] with dropout on the pooled features
        (hidden_0 is then per sample, T = that call's sample count)."""
        width = self.config.hidden_layer_width
        if self._head_T is None:
            raise ValueError("debug_h1 needs a preceding predict")
        shape = (int(n), self._head_T, width) if self.config.dropout_sites[0] else (int(n), width)
        out = np.empty(shape, np.float32)
        _ffi.check(self.ctx.handle, self.lib.bq_model_debug_h1(self.h, int(n), _ffi.ptr(out)), "bq_model_debug_h1")
        return out

    def debug_tags(self) -> list:
        """the `debug_stage` tags of the execution plan, in execution order"""
        buf = C.create_string_buffer(1 << 16)
        _ffi.check(self.ctx.handle, self.lib.bq_model_debug_tags(self.h, buf, len(buf)), "bq_model_debug_tags")
        return buf.value.decode().split()

    KERNEL_FAMILIES = ("tile_stats", "conv1", "gemm_conv2", "gemm_pointwise", "depthwise", "maxpool_add",
                       "subsample", "gap", "head_gemm", "mc_expand", "head_final", "head_fused", "sepconv_fused", "sepconv_mid")

    def set_profiling(self, level: int):
        """0 off, 1 per-stage CUDA-event times, 2 per-kernel-family times + algorithmic work"""
        _ffi.check(self.ctx.handle, self.lib.bq_model_set_profiling(self.h, int(level)), "bq_model_set_profiling")

    def kernel_profile(self):
        """{family: {ms, flops, bytes, launches}} of the last predict() (profiling level 2)"""
        n = 16
        ms, fl, by = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)()
        la = (C.c_int64 * n)()
        _ffi.check(self.ctx.handle, self.lib.bq_model_kernel_profile(self.h, ms, fl, by, la), "bq_model_kernel_profile")
        return {k: dict(ms=ms[i], flops=fl[i], bytes=by[i], launches=int(la[i]))
                for i, k in enumerate(self.KERNEL_FAMILIES)}

    def last_stage_ms(self):
        ms = (C.c_float * 8)()
        _ffi.check(self.ctx.handle, self.lib.bq_model_last_stage_ms(self.h, ms), "bq_model_last_stage_ms")
        names = ("stats+conv1", "conv2", "entry", "middle", "exit", "head")
        return {k: float(ms[i]) for i, k in enumerate(names)}


def predict_table(interface: UncertaintyInterface, tiles, slides, y_true=None, outcome="cohort",
                  T: int | None = None, seed: int = 0, tile_index_base: int = 0, renamed: bool = True):
    """Tile-prediction table for `biscuit_b200.threshold` from raw tiles.

    slides: per-tile slide name; y_true: per-tile label (optional).  With `renamed=True` the columns
    are already the ones `rename_cols` (reference utils.py:31-53) produces (`y_true`, `y_pred`,
    `uncertainty`); otherwise Slideflow's '{outcome}-y_pred1' style headers (utils.py:19-28)."""
    mean, std = interface.predict(tiles, T=T, seed=seed, tile_index_base=tile_index_base)
    cols = {"slide": np.asarray(slides)}
    if y_true is not None:
        cols["y_true" if renamed else y_true_header(outcome)] = np.asarray(y_true)
    cols["y_pred" if renamed else y_pred_header(outcome)] = mean[:, 1]
    cols["uncertainty" if renamed else uncertainty_header(outcome)] = std[:, 1]
    return pd.DataFrame(cols)


def predict_tfrecords(interface: UncertaintyInterface, paths, y_true=None, outcome="cohort", T: int | None = None,
                      seed: int = 0, renamed: bool = True, **keys):
    """`predict_table` straight from Slideflow tile TFRecords: the records of `paths` in file order, JPEG or PNG tiles
    decoded on the GPU.  Tile indices of the dropout streams run across files, so the table equals one `predict_table` over all
    tiles.  y_true: per-tile labels, or a dict slide -> label.  Adds the `loc_x` / `loc_y` columns of each tile.
    `keys` goes to `tfrecord.read`: the feature names (`image_key`, `slide_key`, `x_key`, `y_key`) and the JPEG decode
    options `dct_method` / `fancy_upscaling` (as in `tf.image.decode_jpeg`; `dct_method="INTEGER_FAST"` selects the
    IDCT `decode_jpeg` uses by default, on whose output Slideflow TensorFlow models were trained; ignored for PNG), and
    the PNG decode option `png_convert_rgb` (grayscale, palette, alpha, 16-bit and interlaced PNG tiles converted to
    RGB8 as `decode_png(channels=3)` does; ignored for JPEG)."""
    from . import tfrecord
    batch, slides, loc_x, loc_y = tfrecord.read(paths, **keys)
    if isinstance(y_true, dict):
        y_true = np.asarray([y_true[s] for s in slides])
    df = predict_table(interface, batch, slides, y_true=y_true, outcome=outcome, T=T, seed=seed, renamed=renamed)
    df["loc_x"] = loc_x
    df["loc_y"] = loc_y
    return df
