"""UQ thresholding on the GPU -- drop-in for reference `biscuit.threshold`.

Same call surface, argument meaning, DataFrame mutation and error behaviour as reference
biscuit/threshold.py (`process_tile_predictions` 125-177, `process_group_predictions` 180-245,
`apply` 248-361, `detect` 364-475, `from_cv` 478-557); the arithmetic runs in
libbiscuit_b200.so (csrc/threshold.cu) through the C ABI of include/biscuit_b200.h:

    tile pass              -> bq_tile_process      (error / correct / incorrect / y_pred_bin)
    groupby(level).mean()  -> bq_group_reduce      (row-order Kahan sum in the column dtype)
    roc_curve + Youden + auc -> bq_tile_roc / bq_roc (radix sort + scan, fp64 J, first argmax)
    slide filter + confusion -> bq_group_apply

This module only factorises the string keys, resolves NumPy's scalar-promotion rule for each
comparison and rebuilds the DataFrames.  There is no CPU fallback: without the CUDA library and
a B200 every function raises `NativeLibraryError`.

Deliberate differences from the reference (all documented in DESIGN.md):
  * plotting (`plot=True`) is out of scope and ignored with a warning;
  * ROC curves whose result the reference discards (tile ROC when `tile_pred` is numeric, the
    group ROC when `slide_pred` is numeric) are not computed;
  * a missing y_true / y_pred / uncertainty column raises ValueError (the reference raises
    UnboundLocalError from a bug at threshold.py:184-186).
"""
from __future__ import annotations

import ctypes as C
import logging
import warnings

import numpy as np
import pandas as pd

from . import _ffi, dist as bdist, errors

log = logging.getLogger("biscuit_b200")

_FLOAT_TYPES = (float, np.float16, np.float32, np.float64)   # threshold.py:411
_THRESH_KEYS = ("tile_uq", "slide_uq", "tile_pred", "slide_pred")
_RESULT_KEYS = ("auc", "percent_incl", "acc", "sensitivity", "specificity")


def _is_detect(x) -> bool:
    return isinstance(x, str) and x == "detect"


def _cmp_scalar(t, col_dtype) -> float:
    """The float64 value a column of `col_dtype` is effectively compared with under NumPy >= 2
    promotion (NEP 50), which pandas follows: python scalars are weak (rounded to the column
    dtype first), NumPy scalars are strong (float32 column vs np.float64 compares in float64)."""
    if isinstance(t, (np.floating, np.integer, np.bool_)) or (isinstance(t, np.ndarray) and t.ndim == 0):
        return float(t)
    if col_dtype == np.float32:
        with np.errstate(over="ignore"):
            return float(np.float32(t))
    return float(t)


def _float_col(a: np.ndarray) -> np.ndarray:
    if a.dtype == np.float32 or a.dtype == np.float64:
        return np.ascontiguousarray(a)
    return np.ascontiguousarray(a, dtype=np.float64)


def _label_col(a: np.ndarray, what="y_true") -> np.ndarray:
    """uint8 labels; anything sklearn's roc_curve would reject (non-binary, NaN) -> ValueError."""
    if a.dtype == np.bool_:
        return np.ascontiguousarray(a, dtype=np.uint8)
    with np.errstate(invalid="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        b = a.astype(np.uint8)
    if not np.array_equal(b, a):
        raise ValueError(f"{what}: labels must be 0/1 (continuous / multiclass format is not supported)")
    return np.ascontiguousarray(b)


class _DeviceTable:
    """One tile table resident on the GPU (bq_table) for the duration of a call."""

    def __init__(self, y_pred, uncertainty, y_true, ctx=None):
        self.ctx = ctx or _ffi.default_context()
        self.lib = self.ctx.lib
        yp, un = _float_col(y_pred), _float_col(uncertainty)
        if yp.dtype != un.dtype:       # mixed float widths: promote both (documented deviation)
            yp, un = yp.astype(np.float64), un.astype(np.float64)
        self.dtype = yp.dtype
        self.code = _ffi.BQ_F32 if self.dtype == np.float32 else _ffi.BQ_F64
        self.n = int(yp.shape[0])
        yt = _label_col(y_true)
        if un.shape[0] != self.n or yt.shape[0] != self.n:
            raise ValueError("y_true, y_pred and uncertainty must have the same length")
        h = C.c_void_p()
        _ffi.check(self.ctx.handle,
                   self.lib.bq_table_create(self.ctx.handle, self.n, self.code, _ffi.ptr(yp),
                                            _ffi.ptr(un), _ffi.ptr(yt), C.byref(h)),
                   "bq_table_create")
        self.h = h
        self.n_groups = 0

    def close(self):
        if self.h:
            self.lib.bq_table_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- threshold.py:141 + sklearn input checks
    def validate(self):
        flags = (C.c_int64 * 4)()
        _ffi.check(self.ctx.handle, self.lib.bq_table_validate(self.h, flags), "bq_table_validate")
        return tuple(int(f) for f in flags)

    def tile_process(self, pred_thresh_eff: float, want_columns=True):
        n = self.n
        err = np.empty(n, np.float64) if want_columns else None
        cor = np.empty(n, np.uint8) if want_columns else None
        ybin = np.empty(n, np.uint8) if want_columns else None
        _ffi.check(self.ctx.handle,
                   self.lib.bq_tile_process(self.h, float(pred_thresh_eff), _ffi.ptr(err),
                                            _ffi.ptr(cor), _ffi.ptr(ybin)), "bq_tile_process")
        return err, cor, ybin

    def tile_roc(self, score_sel, label_sel):
        r = _ffi.RocResult()
        _ffi.check(self.ctx.handle, self.lib.bq_tile_roc(self.h, score_sel, label_sel, C.byref(r)),
                   "bq_tile_roc")
        return r

    def set_groups(self, codes: np.ndarray, n_groups: int):
        codes = np.ascontiguousarray(codes, dtype=np.int32)
        _ffi.check(self.ctx.handle, self.lib.bq_table_set_groups(self.h, _ffi.ptr(codes), int(n_groups)),
                   "bq_table_set_groups")
        self.n_groups = int(n_groups)

    def set_filter(self, tile_uq_eff):
        if tile_uq_eff is None:
            rc = self.lib.bq_table_set_tile_filter(self.h, 0, 0.0)
        else:
            rc = self.lib.bq_table_set_tile_filter(self.h, 1, float(tile_uq_eff))
        _ffi.check(self.ctx.handle, rc, "bq_table_set_tile_filter")

    def group_reduce(self):
        L = self.n_groups
        gp, gu = np.empty(L, self.dtype), np.empty(L, self.dtype)
        gt = np.empty(L, np.float64)
        cnt, first = np.empty(L, np.int64), np.empty(L, np.int64)
        _ffi.check(self.ctx.handle,
                   self.lib.bq_group_reduce(self.h, _ffi.ptr(gp), _ffi.ptr(gu), _ffi.ptr(gt),
                                            _ffi.ptr(cnt), _ffi.ptr(first)), "bq_group_reduce")
        return gp, gu, gt, cnt, first


def _roc(ctx, score, label, include=None):
    """bq_roc on host arrays -> RocResult."""
    score = _float_col(np.asarray(score))
    label = np.ascontiguousarray(label, dtype=np.uint8)
    inc = None if include is None else np.ascontiguousarray(include, dtype=np.uint8)
    r = _ffi.RocResult()
    code = _ffi.BQ_F32 if score.dtype == np.float32 else _ffi.BQ_F64
    _ffi.check(ctx.handle,
               ctx.lib.bq_roc(ctx.handle, _ffi.ptr(score), code, _ffi.ptr(label), _ffi.ptr(inc),
                              int(score.shape[0]), C.byref(r)), "bq_roc")
    return r


_EMPTY_INPUT = "Found array with 0 sample(s) while a minimum of 1 is required."   # sklearn's check_array


def _youden_or_raise(r):
    """The reference's `max(zip(tpr,fpr))` / `.index()` idiom raises ValueError for single-class
    labels (SURVEY App. A.1); empty input makes sklearn raise ValueError too."""
    if r.status != 0:
        raise ValueError("(nan, nan) is not in list" if r.status == 1 else _EMPTY_INPUT)
    return np.float64(r.threshold)


def _raise_invalid(n_rows, flags):
    """Raise what the reference raises for a tile table of `n_rows` rows with these `bq_table_validate` counts:
    the NaN check of threshold.py:141, then sklearn's input checks in the first roc_curve."""
    n_nan, n_nonfinite, _, n_badlabel = flags
    if n_nan:
        raise errors.PredsContainNaNError
    if n_nonfinite:
        raise ValueError("Input contains infinity or a value too large for dtype.")
    if n_badlabel:
        raise ValueError("multiclass format is not supported")
    if n_rows == 0:
        raise ValueError(_EMPTY_INPUT)


def _check_columns(df):
    missing = [c for c in ("y_true", "y_pred", "uncertainty") if c not in df.columns]
    if missing:
        raise ValueError("Missing columns. Expected y_true, y_pred, uncertainty. "
                         f"Got: {', '.join(map(str, df.columns))}")


def _factorize(keys: pd.Series):
    codes, uniques = pd.factorize(keys, use_na_sentinel=True)   # first-appearance order, NaN -> -1
    return codes.astype(np.int32, copy=False), uniques


class ResidentTable:
    """A tile-prediction table kept RESIDENT on the GPU across calls.

    The reference re-derives everything from the DataFrame in every call: the nested-CV caller runs `detect` twice per
    inner fold and `apply` twice per outer fold on the same tables (experiment.py:966-1001).  Here the table is
    uploaded once (`bq_table`), and what does not depend on the thresholds being searched is computed once and kept:

      * the tile stage (validation, optional tile-ROC detection of `tile_pred`, the error / correct / incorrect /
        y_pred_bin columns added to the DataFrame, threshold.py:140-177) -- keyed by the `tile_pred` setting;
      * the first-appearance factorisation of the slide / patient keys (threshold.py:190).

    A later call with another tile-UQ threshold only re-runs the filter + reference-order slide reduction and the
    slide-level stage.  `apply_resident` / `detect_resident` are the entry points; `apply` / `detect` are the same code on
    a table that lives for one call, and `apply_sharded` / `detect_sharded` on a :class:`ShardedTable`.  The DataFrame
    is mutated exactly as the reference mutates it.

    `tile_only=True` opens a table for the tile stage alone, which needs no `uncertainty` column
    (`process_tile_predictions`)."""

    def __init__(self, df, ctx=None, tile_only=False):
        if not tile_only:
            _check_columns(df)
        self.df = df
        self.ctx = ctx or _ffi.default_context()
        self.tab = self._open()
        self.dtype = None if self.tab is None else self.tab.dtype
        self.n_unc_nonfinite = 0      # sklearn's finiteness check fires only where the uncertainty feeds a ROC
        self._tile_key = self.pred_thresh = None
        self._keys = {}

    def _open(self):
        df = self.df
        unc = df["uncertainty"].to_numpy() if "uncertainty" in df.columns else np.zeros(len(df), df["y_pred"].to_numpy().dtype)
        return _DeviceTable(df["y_pred"].to_numpy(), unc, df["y_true"].to_numpy(), ctx=self.ctx)

    def close(self):
        if self.tab is not None:
            self.tab.close()
            self.tab = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------------------------
    # tile level
    # ------------------------------------------------------------------------------------
    def tile_stage(self, tile_pred, patients):
        """-> the tile prediction threshold in force (detected once per table when 'detect')."""
        key = "detect" if _is_detect(tile_pred) else (type(tile_pred).__name__, float(tile_pred))
        if key != self._tile_key:
            # a different numeric threshold rewrites the derived columns; the incorrect flags on the device follow
            self.pred_thresh = self._tile_stage(tile_pred, patients)
            self._tile_key = key
        elif patients is not None and "patient" not in self.df.columns:
            self.df["patient"] = self._map_slides(patients)
        return self.pred_thresh

    def _tile_stage(self, pred_thresh, patients):
        """threshold.py:140-177; mutates df; returns pred_thresh used."""
        n_rows, flags = self._validate()
        self.n_unc_nonfinite = flags[2]
        _raise_invalid(n_rows, flags)                                     # :141-142
        if _is_detect(pred_thresh):                                       # :145-159
            r = self._roc_table().tile_roc(_ffi.SCORE_Y_PRED, _ffi.LABEL_Y_TRUE)
            if r.status == 1:
                log.debug("Unable to calculate tile prediction threshold; using 0.5")
                pred_thresh = 0.5                                         # :153-155
            else:
                pred_thresh = _youden_or_raise(r)
            log.debug(f"Auto-detected tile prediction threshold: {pred_thresh:.4f}")
        else:
            log.debug(f"Using tile prediction threshold: {pred_thresh:.4f}")  # :161
        if self.tab is None:                                              # an empty shard is left as it is
            return pred_thresh
        df = self.df
        if patients is not None:                                          # :163-166
            df["patient"] = self._map_slides(patients)
        else:
            log.debug("Patients not provided; assuming 1:1 slide:patient mapping")
        err, cor, ybin = self.tab.tile_process(_cmp_scalar(pred_thresh, df["y_pred"].to_numpy().dtype))
        # dtypes as pandas gives them: |int64 - float| -> float64 (narrow ints keep the float width)
        err_dtype = np.result_type(df["y_true"].to_numpy().dtype, df["y_pred"].to_numpy().dtype)
        df["error"] = err if err_dtype == np.float64 else err.astype(err_dtype)   # :170
        df["correct"] = cor.view(np.bool_)                                # :171-174
        df["incorrect"] = (cor ^ 1).astype(int)                           # :175
        df["y_pred_bin"] = ybin.astype(int)                               # :176
        return pred_thresh

    def _validate(self):
        """-> (rows, bq_table_validate counts) of the table whose errors the reference would raise"""
        return self.tab.n, self.tab.validate()

    def _roc_table(self):
        """the device table the tile-level ROCs run on"""
        return self.tab

    def tile_uq_threshold(self):
        """threshold.py:416-426: Youden's J on the tile ROC of `incorrect ~ uncertainty` (after the tile stage)."""
        if self.n_unc_nonfinite:                                          # roc_curve -> assert_all_finite (uncaught at :419)
            raise ValueError("Input contains NaN or infinity.")
        return _youden_or_raise(self._roc_table().tile_roc(_ffi.SCORE_UNCERTAINTY, _ffi.LABEL_INCORRECT))

    def _map_slides(self, patients):
        """``df['slide'].map(patients)`` computed on the UNIQUE slide names and expanded through the factorisation
        codes (same `Series.map` on the same values, so the same dtype inference and NaN for unknown slides), instead
        of a hash lookup per tile row; the factorisation is the one the slide-level grouping uses."""
        df = self.df
        codes, uniques = self.keys("slide")
        if len(codes) == 0 or codes.min() < 0:                            # NaN slide names: leave it to pandas
            return df["slide"].map(patients)
        mapped = pd.Series(uniques, dtype=df["slide"].dtype).map(patients)
        return pd.Series(mapped.array.take(codes), index=df.index)

    # ------------------------------------------------------------------------------------
    # group (slide / patient) level
    # ------------------------------------------------------------------------------------
    def keys(self, level):
        """(codes, uniques) of df[level] in first-appearance order, factorised once per level"""
        if level not in self._keys:
            self._keys[level] = _factorize(self.df[level])
        return self._keys[level]

    def _reduce(self, level, tile_uq_eff):
        """threshold.py:190-192 with the tile-UQ filter: -> (keys, number of keys before the filter with NaN counted as
        one, per-key (y_pred, uncertainty, y_true) means, surviving tile counts and first surviving rows)"""
        codes, uniques = self.keys(level)
        self.tab.set_groups(codes, len(uniques))
        self.tab.set_filter(tile_uq_eff)
        return uniques, len(uniques) + int((codes < 0).any()), self.tab.group_reduce()

    def _groups(self, level, tile_uq_eff):
        """-> (keys, y_pred, uncertainty, y_true truncated to uint8, keys before the filter) of the groups with a
        surviving tile, in first-appearance order after the filter"""
        uniques, n_keys, (gp, gu, gt, cnt, first) = self._reduce(level, tile_uq_eff)
        alive = np.flatnonzero(cnt > 0)
        order = alive[np.argsort(first[alive], kind="stable")]
        return [uniques[i] for i in order], gp[order], gu[order], gt[order].astype(np.uint8), n_keys

    def group_table(self, level, tile_uq_eff, pred_thresh):
        """threshold.py:188-245 with the tile-UQ filter (threshold.py:298/412/426) applied on the device: the per-group
        means (:190-200), optional Youden detection on the group ROC, then the group DataFrame.
        -> (group DataFrame, pred_thresh used, number of keys before the filter)"""
        levels, yp, u, yt, n_keys = self._groups(level, tile_uq_eff)
        if not len(yt):                                                   # :205-206
            raise errors.ROCFailedError("Unable to generate ROC; preds are empty.")
        if _is_detect(pred_thresh):                                       # :217-223
            r = _roc(self.ctx, yp, yt)
            if r.status != 0:
                raise errors.ROCFailedError(f"Unable to generate {level}-level ROC")
            pred_thresh = np.float64(r.threshold)
            log.debug(f"Using detected prediction threshold: {pred_thresh:.4f}")
        else:
            log.debug(f"Using {level} prediction threshold: {pred_thresh:.4f}")   # :225
        cols = _group_columns(self.ctx, yp, u, yt, pred_thresh, pred_thresh, _ffi.KEEP_ALL, 0.0)
        l_df = pd.DataFrame({                                             # :235-244
            level: pd.Series(levels),
            "error": pd.Series(cols["error"]),
            "uncertainty": pd.Series(u),
            "correct": cols["correct"].view(np.bool_),
            "incorrect": pd.Series(cols["incorrect"]).astype(int),
            "y_true": pd.Series(yt),
            "y_pred": pd.Series(yp),
            "y_pred_bin": pd.Series(cols["y_pred_bin"].view(np.bool_)).astype(int),
        })
        return l_df, pred_thresh, n_keys


class ShardedTable(ResidentTable):
    """This rank's shard of a cohort sharded over ranks (SURVEY.md 8e): one process per GPU, torch.distributed
    initialised or a `dist.NativeComm` passed as `group`.  Every rank holds a contiguous, slide-aligned shard of the tile
    table (see `dist.shard_bounds`; a slide / patient must not straddle ranks; a shard may be empty) and runs the same
    calls in the same order, so every rank makes the same collectives:

      * validation counts are summed over the ranks, so every rank raises what the concatenated table raises (a rank
        that raised alone would leave the others blocked in a collective);
      * the tile-level ROCs run over ALL tiles of the cohort: the per-tile `(pred, unc, label)` triples are all-gathered
        into a second `bq_table` on every GPU (deterministic kernels: replicated, identical thresholds);
      * tile processing and the reference-order per-group reduction stay local and bit-exact; the per-group aggregates
        and names are all-gathered (`dist.all_gather_groups`) and the group level runs replicated.

    An empty shard opens no `bq_table` and contributes zero groups."""

    def __init__(self, df, group=None):
        self.group, self.cohort = group, None
        self.rows, self.cohort_dtype = [], None        # every rank's row count and the cohort dtype, from the validation
        super().__init__(df)
        self.device = f"cuda:{self.ctx.device}"

    def _open(self):
        return super()._open() if len(self.df) else None

    def close(self):
        super().close()
        if self.cohort is not None:
            self.cohort.close()
            self.cohort = None

    def _validate(self):
        n_rows, flags = super()._validate() if self.tab is not None else (0, (0, 0, 0, 0))
        dcode = -1 if self.dtype is None else int(self.dtype == np.float64)
        meta = bdist.all_gather_meta([n_rows, dcode, *flags], group=self.group, device=self.device)
        self.rows = [int(n) for n in meta[:, 0]]
        self.cohort_dtype = np.dtype(np.float64 if (meta[:, 1] == 1).any() else np.float32)
        return sum(self.rows), tuple(int(f) for f in meta[:, 2:].sum(axis=0))

    def _roc_table(self):
        if self.cohort is None:
            dt, df = self.cohort_dtype, self.df
            buf = bdist.pack_tiles(_float_col(df["y_pred"].to_numpy()).astype(dt, copy=False),
                                   _float_col(df["uncertainty"].to_numpy()).astype(dt, copy=False),
                                   _label_col(df["y_true"].to_numpy()))
            parts = bdist.all_gather_bytes(buf, [n * (2 * dt.itemsize + 1) for n in self.rows],
                                           group=self.group, device=self.device)
            cols = [bdist.unpack_tiles(part, n, dt) for n, part in zip(self.rows, parts)]
            self.cohort = _DeviceTable(*(np.concatenate(c) for c in zip(*cols)), ctx=self.ctx)
        return self.cohort

    def tile_uq_threshold(self):
        cohort = self._roc_table()
        cohort.tile_process(_cmp_scalar(self.pred_thresh, cohort.dtype), want_columns=False)   # its incorrect flags
        return super().tile_uq_threshold()

    def _groups(self, level, tile_uq_eff):
        names, n_keys, local = [], 0, (np.zeros(0),) * 5
        if self.tab is not None:
            uniques, n_keys, local = self._reduce(level, tile_uq_eff)
            names = [str(u) for u in uniques]
        g, names, n_keys = bdist.all_gather_groups(names, local, len(self.df), n_keys, self.cohort_dtype,
                                                   group=self.group, device=self.device)
        return [names[c] for c in g["code"]], g["y_pred"], g["uncertainty"], g["y_true"], n_keys


def process_tile_predictions(df, pred_thresh=0.5, patients=None):
    """Tile-level processing (reference threshold.py:125-177).

    Adds `error`, `correct`, `incorrect`, `y_pred_bin` (and `patient`) to `df` IN PLACE and returns
    ``(df, pred_thresh)``; ``pred_thresh='detect'`` picks Youden's J on the tile ROC."""
    with ResidentTable(df, tile_only=True) as table:
        return df, table.tile_stage(pred_thresh, patients)


def _group_columns(ctx, yp, u, yt, pred_thresh, strict_thresh, keep_mode, slide_uq_eff):
    L = int(yp.shape[0])
    dt = yp.dtype
    code = _ffi.BQ_F32 if dt == np.float32 else _ffi.BQ_F64
    out = {"error": np.empty(L, dt), "correct": np.empty(L, np.uint8), "incorrect": np.empty(L, np.uint8),
           "y_pred_bin": np.empty(L, np.uint8), "include": np.empty(L, np.uint8)}
    conf = (C.c_int64 * 4)()
    yp, u, yt = np.ascontiguousarray(yp), np.ascontiguousarray(u), np.ascontiguousarray(yt)
    _ffi.check(ctx.handle,
               ctx.lib.bq_group_apply(ctx.handle, L, code, _ffi.ptr(yp), _ffi.ptr(u), _ffi.ptr(yt),
                                      _cmp_scalar(pred_thresh, dt), _cmp_scalar(strict_thresh, dt),
                                      int(keep_mode), float(slide_uq_eff),
                                      _ffi.ptr(out["error"]), _ffi.ptr(out["correct"]),
                                      _ffi.ptr(out["incorrect"]), _ffi.ptr(out["y_pred_bin"]),
                                      _ffi.ptr(out["include"]), conf), "bq_group_apply")
    out["confusion"] = tuple(np.int64(c) for c in conf)
    return out


def process_group_predictions(df, pred_thresh, level):
    """Group-level (slide / patient) predictions and uncertainty from tile-level rows
    (reference threshold.py:180-245): per-group means in first-appearance order, `y_true`
    truncated to uint8, `correct / incorrect / y_pred_bin` with ``>= pred_thresh``.
    ``pred_thresh='detect'`` picks Youden's J on the group ROC (ROCFailedError if impossible)."""
    _check_columns(df)
    if len(df) == 0:
        df[level]                                                     # KeyError parity
        raise errors.ROCFailedError("Unable to generate ROC; preds are empty.")
    with ResidentTable(df) as table:
        return table.group_table(level, None, pred_thresh)[:2]


def _auc_included(ctx, s_yp, s_yt, include=None):
    """utils.py:487-504: ROC AUC of the surviving groups, NaN when undefined."""
    r = _roc(ctx, s_yp, s_yt, include)
    if r.status == 2:
        log.warning("Unable to calculate ROC")
        return np.nan
    return float(r.auc)


def _apply_preamble(df, tile_uq, keep, patients, level):
    """threshold.py:281-287, before the table is opened."""
    assert keep in ("high_confidence", "low_confidence")             # :281
    assert not (level == "patient" and patients is None)             # :282
    log.debug(f"Applying tile UQ threshold of {tile_uq:.5f}")         # :284 (TypeError on None)
    if patients:                                                      # :285-286
        df["patient"] = df["slide"].map(patients)
    df[level]                                                         # :287 KeyError parity


def apply(df, tile_uq, slide_uq, tile_pred=0.5, slide_pred=0.5, plot=False,
          keep="high_confidence", title=None, patients=None, level="slide"):
    """Apply pre-calculated tile- and group-level uncertainty thresholds
    (reference threshold.py:248-361).

    Args:
        df (pandas.DataFrame): columns 'y_true', 'y_pred', 'uncertainty', 'slide'. Mutated in place
            exactly like the reference (adds error / correct / incorrect / y_pred_bin / patient).
        tile_uq (float): tile-level uncertainty threshold (falsy: no tile filter).
        slide_uq (float): group-level uncertainty threshold (falsy: no group filter).
        tile_pred, slide_pred (float): prediction thresholds. Default 0.5.
        keep (str): 'high_confidence' (uncertainty < slide_uq) or 'low_confidence' (>=).
        patients (dict): slide -> patient; required for level='patient'.
        level (str): 'slide' or 'patient'.

    Returns:
        dict with auc, percent_incl, acc, sensitivity, specificity; DataFrame of the kept groups
        (original integer index labels).  ({...None}, None) if no group-level ROC is possible."""
    if plot:
        log.warning("plot=True ignored: plotting is outside the scope of biscuit_b200")
    _apply_preamble(df, tile_uq, keep, patients, level)
    with ResidentTable(df) as table:
        return apply_resident(table, tile_uq, slide_uq, tile_pred=tile_pred, slide_pred=slide_pred, keep=keep,
                              patients=patients, level=level)


def apply_resident(table: ResidentTable, tile_uq, slide_uq, tile_pred=0.5, slide_pred=0.5, plot=False,
                   keep="high_confidence", title=None, patients=None, level="slide"):
    """`apply` on a table that is already resident on the GPU (see :class:`ResidentTable`): the tile stage and the key
    factorisation are reused from earlier calls, only the filter + slide reduction + slide-level stage run."""
    assert keep in ("high_confidence", "low_confidence")
    assert not (level == "patient" and patients is None)
    df = table.df
    if patients and "patient" not in df.columns:
        df["patient"] = df["slide"].map(patients)
    df[level]
    table.tile_stage(tile_pred, patients)                             # :290-294
    tile_uq_eff = _cmp_scalar(tile_uq, table.dtype) if tile_uq else None   # :297-298
    try:
        s_df, _, n_before = table.group_table(level, tile_uq_eff, slide_pred)   # :295, :305
    except errors.ROCFailedError:
        log.error("Unable to process slide predictions")
        return {k: None for k in _RESULT_KEYS}, None                  # :310-317
    return _apply_group_level(table.ctx, s_df, slide_uq, slide_pred, keep, level, n_before)


def _apply_group_level(ctx, s_df, slide_uq, slide_pred, keep, level, n_before):
    """threshold.py:323-361: group-level UQ filter, AUROC, percent included and the confusion counts."""
    yp, u, yt = s_df["y_pred"].to_numpy(), s_df["uncertainty"].to_numpy(), s_df["y_true"].to_numpy()
    if slide_uq:                                                      # :323-330
        log.debug(f"Using {level} uncertainty threshold of {slide_uq:.5f}")
        mode = _ffi.KEEP_HIGH if keep == "high_confidence" else _ffi.KEEP_LOW
        uq_eff = _cmp_scalar(slide_uq, u.dtype)
    else:
        mode, uq_eff = _ffi.KEEP_ALL, 0.0
    cols = _group_columns(ctx, yp, u, yt, slide_pred, slide_pred, mode, uq_eff)
    include = cols["include"].view(np.bool_)
    if slide_uq:
        s_df = s_df.loc[include]
    auc = _auc_included(ctx, yp, yt, cols["include"])                 # :333
    percent_incl = len(s_df) / n_before                               # :334-335
    tp, fp, tn, fn = cols["confusion"]                                # :339-345
    with np.errstate(invalid="ignore", divide="ignore"):
        results = {"auc": auc, "percent_incl": percent_incl,
                   "acc": (tp + tn) / (tp + tn + fp + fn),            # :346
                   "sensitivity": tp / (tp + fn),                     # :347
                   "specificity": tn / (tn + fp)}                     # :348
    return results, s_df


def apply_sharded(df, tile_uq, slide_uq, tile_pred=0.5, slide_pred=0.5, keep="high_confidence",
                  patients=None, level="slide", group=None):
    """`apply` for a cohort sharded over ranks: every rank passes ITS shard of the tile table (see
    :class:`ShardedTable`) and returns the same (results, s_df) `apply` would return on the concatenated table, or
    raises the same exception.  Thresholds must be numeric: 'detect' is resolved on the whole cohort by
    `detect_sharded`."""
    if _is_detect(tile_pred) or _is_detect(slide_pred):
        raise ValueError("apply_sharded needs numeric prediction thresholds (a per-shard 'detect' would differ "
                         "between ranks): use detect_sharded / from_cv_sharded first")
    _apply_preamble(df, tile_uq, keep, patients, level)
    with ShardedTable(df, group=group) as table:
        return apply_resident(table, tile_uq, slide_uq, tile_pred=tile_pred, slide_pred=slide_pred, keep=keep,
                              patients=patients, level=level)


def detect(df, tile_uq="detect", slide_uq="detect", tile_pred="detect", slide_pred="detect",
           plot=False, patients=None):
    """Detect optimal tile- and slide-level uncertainty thresholds (reference threshold.py:364-475).

    Each of tile_uq / slide_uq / tile_pred / slide_pred is 'detect' (Youden's J on the matching
    ROC) or a float to use as given.  Returns (dict of the four thresholds, slide-level AUROC), or
    (all-None dict, None) when predictions contain NaN or no slide-level ROC is possible."""
    if plot:
        log.warning("plot=True ignored: plotting is outside the scope of biscuit_b200")
    with ResidentTable(df) as table:
        return detect_resident(table, tile_uq=tile_uq, slide_uq=slide_uq, tile_pred=tile_pred, slide_pred=slide_pred,
                               patients=patients)


def detect_resident(table: ResidentTable, tile_uq="detect", slide_uq="detect", tile_pred="detect", slide_pred="detect",
                    plot=False, patients=None):
    """`detect` on a GPU-resident table (see :class:`ResidentTable`) or on this rank's :class:`ShardedTable`."""
    none4 = {k: None for k in _THRESH_KEYS}
    try:
        found_tile_pred = table.tile_stage(tile_pred, patients)       # :398-402
    except errors.PredsContainNaNError:
        log.error("Tile-level predictions contain NaNs; unable to process.")
        return none4, None                                            # :403-405
    if _is_detect(tile_pred):                                         # :407-408
        tile_pred = found_tile_pred
    if isinstance(tile_uq, _FLOAT_TYPES):                             # :411-412
        tile_uq_eff = _cmp_scalar(tile_uq, table.dtype)
    elif not _is_detect(tile_uq):                                     # :413-415
        log.debug("Not performing tile-level uncertainty thresholding.")
        tile_uq, tile_uq_eff = None, None
    else:                                                             # :416-426
        tile_uq = table.tile_uq_threshold()
        log.debug(f"Tile-level optimal UQ threshold: {tile_uq:.4f}")
        tile_uq_eff = float(tile_uq)
    try:
        s_df, slide_pred, _ = table.group_table("slide", tile_uq_eff, slide_pred)   # :433-438
    except errors.ROCFailedError:
        log.error("Unable to process slide predictions")
        return none4, None                                            # :439-441
    slide_uq, auc = _detect_group_level(table.ctx, s_df, slide_uq, slide_pred)
    return {"tile_uq": tile_uq, "slide_uq": slide_uq,
            "tile_pred": tile_pred, "slide_pred": slide_pred}, auc


def _detect_group_level(ctx, s_df, slide_uq, slide_pred):
    """threshold.py:444-468: slide-level UQ threshold (Youden on incorrect ~ uncertainty) and the AUROC of the kept slides."""
    yp, u, yt = s_df["y_pred"].to_numpy(), s_df["uncertainty"].to_numpy(), s_df["y_true"].to_numpy()
    include = None
    if _is_detect(slide_uq):                                          # :444-460
        inc = s_df["incorrect"].to_numpy()
        if not inc.sum():
            log.debug("Unable to calculate slide UQ threshold; no incorrect predictions made")
            slide_uq = None
        else:
            slide_uq = _youden_or_raise(_roc(ctx, u, inc))
            log.debug(f"Slide-level optimal UQ threshold: {slide_uq:.4f}")
            include = _group_columns(ctx, yp, u, yt, slide_pred, slide_pred, _ffi.KEEP_HIGH,
                                     float(slide_uq))["include"]
    else:
        log.debug("Not performing slide-level uncertainty thresholding.")
        slide_uq = 0.5                                                # :461-463
    return slide_uq, _auc_included(ctx, yp, yt, include)              # :468


def detect_sharded(df, tile_uq="detect", slide_uq="detect", tile_pred="detect", slide_pred="detect",
                   patients=None, group=None):
    """`detect` for a table sharded over ranks (see :class:`ShardedTable`): the reference's threshold.py:364-475 on the
    concatenated table, with the tile-level ROCs over all tiles of the cohort.  Returns what `detect` returns, on every
    rank."""
    with ShardedTable(df, group=group) as table:
        return detect_resident(table, tile_uq=tile_uq, slide_uq=slide_uq, tile_pred=tile_pred, slide_pred=slide_pred,
                               patients=patients)


def from_cv(dfs, **kwargs):
    """Optimal tile- and slide-level thresholds from a set of (nested) cross-validation folds
    (reference threshold.py:478-557): `detect` per fold, folds without a tile_uq / slide_uq are
    skipped, then tile_uq = min, slide_uq = max, tile_pred / slide_pred = mean over folds.

    Args:
        dfs (list(DataFrame)): tile predictions with 'y_true', 'y_pred', 'uncertainty', 'slide',
            'patient'.
        **kwargs: forwarded to :func:`detect` (tile_uq, slide_uq, tile_pred, slide_pred, patients).

    Raises ValueError for missing columns and ThresholdError when no fold yields a threshold."""
    return _from_cv(dfs, detect, kwargs)


def from_cv_sharded(dfs, group=None, **kwargs):
    """`from_cv` with every fold table sharded over the ranks: `detect_sharded` per fold, same fold-skipping and
    min / max / mean reduction over folds as the reference (threshold.py:478-557)."""
    return _from_cv(dfs, lambda df, **kw: detect_sharded(df, group=group, **kw), kwargs, require_patient=False)


class FoldSet:
    """The tile tables of a set of cross-validation folds, uploaded once and kept resident on the GPU.

    `from_cv` may then be called repeatedly -- the nested-CV caller detects the tile-level UQ threshold first and the
    slide-level thresholds with that tile threshold fixed (reference experiment.py:966-977) -- and every call after the
    first reuses each fold's tile stage and key factorisation (:class:`ResidentTable`)."""

    def __init__(self, dfs, ctx=None):
        self.tables = []
        try:
            for df in dfs:
                missing = [c for c in _CV_COLUMNS if c not in df.columns]
                if missing:
                    raise ValueError(f"DataFrame missing columns, expected {_CV_COLUMNS}, got: "
                                     f"{', '.join(df.columns.tolist())}")
                self.tables.append(ResidentTable(df, ctx=ctx))
        except Exception:
            self.close()
            raise

    def close(self):
        for t in self.tables:
            t.close()
        self.tables = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __len__(self):
        return len(self.tables)

    def from_cv(self, **kwargs):
        """same result as ``threshold.from_cv([t.df for t in tables], **kwargs)`` (reference threshold.py:478-557)"""
        return _from_cv(self.tables, lambda t, **kw: detect_resident(t, **kw), kwargs, columns_of=lambda t: t.df.columns)


_CV_COLUMNS = ("y_true", "y_pred", "uncertainty", "slide", "patient")


def _from_cv(dfs, detect_fn, kwargs, require_patient=True, columns_of=lambda df: df.columns):
    """Fold pass + reduction of the reference's from_cv (threshold.py:478-557): every fold table is validated and run
    through `detect_fn`; folds without both UQ thresholds drop out (:526-528); the survivors reduce to
    min(tile_uq), max(slide_uq), mean(tile_pred), mean(slide_pred) (:544-557).  The two `*_uq_thresh=None` keywords
    switch a UQ reduction off and leave an empty list in its place, as the reference does (:513-516)."""
    required = ("y_true", "y_pred", "uncertainty", "slide") + (("patient",) if require_patient else ())
    kept = []
    for idx, df in enumerate(dfs):
        log.debug(f"Detecting thresholds from fold {idx}")
        present = list(columns_of(df))
        if any(col not in present for col in required):
            raise ValueError(f"DataFrame missing columns, expected {required}, got: {', '.join(present)}")
        fold, _ = detect_fn(df, **kwargs)
        if fold["tile_uq"] is None or fold["slide_uq"] is None:
            log.debug(f"Skipping CV #{idx}, unable to detect threshold")
            continue
        kept.append(fold)
    reducers = {"tile_uq": ("tile", np.min), "slide_uq": ("slide", np.max)}
    out = {}
    for key, (what, reduce_fn) in reducers.items():
        switched_off = kwargs.get(f"{key}_thresh", 0) is None and f"{key}_thresh" in kwargs
        if switched_off:
            out[key] = []
        elif not kept:
            raise errors.ThresholdError(f"Unable to detect {what} UQ threshold.")
        else:
            out[key] = reduce_fn([fold[key] for fold in kept])
    for key in ("tile_pred", "slide_pred"):
        out[key] = np.mean([fold[key] for fold in kept])
    return out
