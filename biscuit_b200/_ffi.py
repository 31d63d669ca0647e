"""ctypes binding of libbiscuit_b200.so (the C ABI declared in include/biscuit_b200.h).

Loading is lazy so that `import biscuit_b200` works on a box without a GPU (the CPU test tier checks
symbols only); any compute call without the library / a GPU raises NativeLibraryError -- there is
deliberately no fallback implementation.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from .errors import NativeLibraryError

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libbiscuit_b200.so")

BQ_F32, BQ_F64 = 0, 1
SCORE_Y_PRED, SCORE_UNCERTAINTY = 0, 1
LABEL_Y_TRUE, LABEL_INCORRECT = 0, 1
KEEP_ALL, KEEP_HIGH, KEEP_LOW = 0, 1, 2

c_void_pp = C.POINTER(C.c_void_p)


class RocResult(C.Structure):
    _fields_ = [("threshold", C.c_double), ("youden_j", C.c_double), ("auc", C.c_double),
                ("n_pos", C.c_int64), ("n_neg", C.c_int64), ("n_points", C.c_int64),
                ("best_index", C.c_int64), ("status", C.c_int32), ("auc_exact", C.c_int32)]


class ModelConfig(C.Structure):
    _fields_ = [("tile_px", C.c_int32), ("hidden_width", C.c_int32), ("hidden_layers", C.c_int32),
                ("n_classes", C.c_int32), ("dropout", C.c_float), ("max_batch", C.c_int32),
                ("dropout_sites", C.c_int32), ("reserved", C.c_int32 * 7)]


class NamedTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int32),
                ("shape", C.c_int64 * 4)]


# name -> (restype, argtypes); every symbol include/biscuit_b200.h declares
SIGNATURES = {
    "bq_abi_version": (C.c_int, []),
    "bq_create": (C.c_int, [C.c_int, c_void_pp]),
    "bq_destroy": (None, [C.c_void_p]),
    "bq_last_error": (C.c_char_p, [C.c_void_p]),
    "bq_launch_count": (C.c_int64, [C.c_void_p]),
    "bq_sync": (C.c_int, [C.c_void_p]),
    "bq_stream": (C.c_void_p, [C.c_void_p]),
    "bq_heatmap_build": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p]),
    "bq_heatmap_mask": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    "bq_comm_unique_id": (C.c_int, [C.c_void_p]),
    "bq_comm_init": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "bq_comm_size": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "bq_comm_destroy": (None, [C.c_void_p]),
    "bq_allgather_bytes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "bq_table_create": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p, c_void_pp]),
    "bq_table_destroy": (None, [C.c_void_p]),
    "bq_table_set_groups": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "bq_table_validate": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "bq_tile_process": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bq_tile_roc": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(RocResult)]),
    "bq_roc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                         C.POINTER(RocResult)]),
    "bq_table_set_tile_filter": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "bq_group_reduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "bq_group_apply": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_double, C.c_double, C.c_int, C.c_double, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.POINTER(C.c_int64)]),
    "bq_model_create": (C.c_int, [C.c_void_p, C.POINTER(ModelConfig), c_void_pp]),
    "bq_model_destroy": (None, [C.c_void_p]),
    "bq_model_load_weights": (C.c_int, [C.c_void_p, C.POINTER(NamedTensor), C.c_int32]),
    "bq_predict_uq": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64,
                                C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bq_predict_uq_standardized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64,
                                             C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bq_model_debug_stage": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_char_p, C.c_void_p,
                                       C.c_int64, C.POINTER(C.c_int64)]),
    "bq_model_debug_h1": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "bq_model_debug_tags": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "bq_stain_normalize": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "bq_model_set_normalizer": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "bq_bootstrap_confusion": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32,
                                         C.c_void_p]),
    "bq_delong_placements": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "bq_model_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "bq_model_last_stage_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "bq_debug_umma_probe": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bq_model_kernel_profile": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                          C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "bq_jpeg_status_string": (C.c_char_p, [C.c_int32]),
    "bq_jpeg_inspect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "bq_jpeg_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "bq_jpeg_last_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "bq_predict_uq_jpeg": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bq_png_status_string": (C.c_char_p, [C.c_int32]),
    "bq_png_inspect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "bq_png_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "bq_predict_uq_png": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bq_tfrecord_scan": (C.c_int, [C.c_void_p, C.c_int64, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int64,
                                   C.POINTER(C.c_int64), C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int64]),
    "bq_crc32c": (C.c_uint32, [C.c_void_p, C.c_int64]),
    "bq_crc32c_masked": (C.c_uint32, [C.c_void_p, C.c_int64]),
}

BQ_ERR_DATA = -6

_lib = None
_lock = threading.Lock()


def load_library():
    """dlopen the in-tree library and bind every symbol.  Does NOT need a GPU."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} not found. Build it with `python -m biscuit_b200.build` "
                "(nvcc, sm_100a). biscuit_b200 has no CPU fallback.")
        try:
            lib = C.CDLL(LIB_PATH)
        except OSError as e:
            raise NativeLibraryError(f"failed to load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:
                raise NativeLibraryError(f"{LIB_PATH} does not export {name}") from e
            fn.restype = res
            fn.argtypes = args
        if lib.bq_abi_version() != 1:
            raise NativeLibraryError("ABI version mismatch between _ffi.py and libbiscuit_b200.so")
        _lib = lib
        return lib


def check(ctx_handle, rc, what=""):
    """raise on a failing return code: ValueError for malformed input data (BQ_ERR_DATA), else NativeLibraryError"""
    if rc == 0:
        return
    lib = load_library()
    msg = lib.bq_last_error(ctx_handle)
    msg = msg.decode() if msg else ""
    if rc == BQ_ERR_DATA:
        raise ValueError(msg)
    raise NativeLibraryError(f"{what or 'libbiscuit_b200 call'} failed (rc={rc}): {msg}")


class Context:
    """One bq_ctx (one GPU, one host thread)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.bq_create(int(device), C.byref(h))
        if rc != 0:
            msg = self.lib.bq_last_error(None)
            raise NativeLibraryError(
                f"bq_create(device={device}) failed (rc={rc}): {msg.decode() if msg else ''} "
                "-- biscuit_b200 needs a B200 (sm_100a); there is no CPU fallback.")
        self.handle = h
        self.device = int(device)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.bq_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(self.lib.bq_launch_count(self.handle))

    @property
    def stream(self) -> int:
        return int(self.lib.bq_stream(self.handle) or 0)

    def sync(self):
        check(self.handle, self.lib.bq_sync(self.handle), "bq_sync")


_default_ctx = {}


def default_context(device: int | None = None) -> Context:
    """Process-wide context per device (device defaults to LOCAL_RANK, else 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    key = (os.getpid(), threading.get_ident(), device)
    ctx = _default_ctx.get(key)
    if ctx is None:
        ctx = Context(device)
        _default_ctx[key] = ctx
    return ctx


def ptr(a):
    """Raw pointer of a numpy array / torch tensor / None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(f"cannot take a pointer of {type(a)}")
