"""Shared test helpers: golden decoding, bit-exact DataFrame / scalar comparison, degenerate tiles."""
import hashlib
import json
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name="threshold_golden.json"):
    with open(os.path.join(GOLDEN_DIR, name)) as f:
        return json.load(f)


def dec(v):
    if v is None:
        return None
    if "hex" in v:
        x = float.fromhex(v["hex"])
        return np.float64(x) if v["t"] == "float64" else (np.float32(x) if v["t"] == "float32" else x)
    return np.int64(v["int"]) if v["t"] != "int" else v["int"]


def same_scalar(a, b, check_type=True):
    if a is None or b is None:
        return a is None and b is None
    if check_type and type(a) is not type(b):
        return False
    return bool(a == b) or (a != a and b != b)


def df_sha(df):
    """same digest as oracle/make_golden.py:enc_df"""
    h = hashlib.sha256()
    h.update(np.asarray(df.index, dtype=np.int64).tobytes())
    for c in df.columns:
        a = df[c].to_numpy()
        if a.dtype.kind in "OUT" or str(df[c].dtype) == "str":
            h.update("|".join(str(x) for x in a).encode())
        else:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def assert_same_df(a, b, what=""):
    if a is None or b is None:
        assert a is None and b is None, f"{what}: one side is None"
        return
    assert list(a.columns) == list(b.columns), f"{what}: columns {list(a.columns)} vs {list(b.columns)}"
    assert a.index.equals(b.index), f"{what}: index differs"
    for c in a.columns:
        assert a[c].dtype == b[c].dtype, f"{what}: dtype of {c}: {a[c].dtype} vs {b[c].dtype}"
        x, y = a[c].to_numpy(), b[c].to_numpy()
        if x.dtype.kind == "f":
            assert np.array_equal(x, y, equal_nan=True), f"{what}: column {c} differs"
            assert x.tobytes() == y.tobytes() or np.isnan(x).any(), f"{what}: column {c} bits differ"
        else:
            assert (x == y).all(), f"{what}: column {c} differs"


def assert_same_results(a, b, what=""):
    assert set(a) == set(b), what
    for k in a:
        assert same_scalar(a[k], b[k]), f"{what}: {k}: {a[k]!r} ({type(a[k]).__name__}) vs {b[k]!r} ({type(b[k]).__name__})"


def degenerate_tiles():
    """4 tiles with large uniform regions (all-zero channels deep in the net)"""
    t = np.zeros((4, 299, 299, 3), np.uint8)
    t[0] = 255                                                          # white background
    t[1] = 237                                                          # constant, odd value
    t[2] = 200; t[2, 150, 150, 1] = 201                                 # a single pixel differs
    t[3] = (np.indices((299, 299)).sum(0) % 2 * 255).astype(np.uint8)[..., None]   # checkerboard 0 / 255
    return t


def tf_standardize(tiles_u8):
    """tf.image.per_image_standardization in numpy fp32: (x - mean) / max(std, 1 / sqrt(N)), a division (TF divides; the
    oracle multiplies by the reciprocal)"""
    x = tiles_u8.astype(np.float32)
    n = np.float32(x[0].size)
    m = x.mean((1, 2, 3), dtype=np.float32, keepdims=True)
    var = np.maximum((x * x).mean((1, 2, 3), dtype=np.float32, keepdims=True) - m * m, np.float32(0))
    sd = np.maximum(np.sqrt(var), np.float32(1) / np.sqrt(n))
    return ((x - m) / sd).astype(np.float32)


def float_tile_sets(weights):
    """name -> 8 float32 NHWC tiles for the route of already-standardised input (`predict` on float32); in each set the
    first four tiles are synthetic and the last four degenerate, except where noted"""
    from oracle import synth, xception_uq as X
    deg = degenerate_tiles()
    u8 = [np.concatenate([synth.tiles_u8(4, seed=s, n_slides=2), deg]) for s in (0, 1, 2)]
    nhwc = lambda t: t.permute(0, 2, 3, 1).contiguous().numpy()             # noqa: E731
    rng = np.random.default_rng(7)
    big = np.empty((8, 299, 299, 3), np.float32)
    big[:4] = rng.uniform(-1e4, 1e4, (4, 299, 299, 3))                      # |x| up to 1e4
    big[4:6] = np.where(rng.random((2, 299, 299, 3)) < 0.5, -1e4, 1e4)      # exactly +-1e4
    big[6], big[7] = 1e4, -1e4                                              # constant
    return {
        # the oracle's (x - mean) * (1 / std): a constant tile becomes exact zeros, the single-pixel tile an outlier of ~518
        "oracle": nhwc(X.XceptionUQOracle(weights).standardize(u8[0])),
        "tf": tf_standardize(u8[1]),
        "raw": u8[2].astype(np.float32),                                    # legal input, not standardised
        "big": big,
    }
