"""GPU tier of TensorFlow's decode_jpeg options: the CUDA decoder with dct_method="INTEGER_FAST" and
fancy_upscaling=False equals libjpeg-turbo's IFAST decode (Pillow's draft route) byte for byte over the quality x
sampling x restart x tile matrix, the other two non-default combinations equal the numpy restatement, the options
apply per call on a reused context, and `predict` / `predict_tfrecords` decode with them."""
import ctypes as C
import itertools

import numpy as np
import pytest

from biscuit_b200 import _ffi, jpeg, threshold, uq
from biscuit_b200.jpeg import JpegBatch
from jpeg_fast_ref import decode as ref_decode
from jpeg_fast_ref import dqt16_encode, pil_decode_fast, saturated_tiles
from oracle import jpeg_synth, synth

pytestmark = pytest.mark.gpu

QUALITIES = (1, 10, 25, 50, 75, 90, 95, 100)
SAMPLINGS = ("4:4:4", "4:2:2", "4:2:0")
RESTARTS = ({}, {"restart_blocks": 1}, {"restart_blocks": 7}, {"restart_rows": 1})
FAST = dict(dct_method="INTEGER_FAST", fancy_upscaling=False)


@pytest.fixture(scope="module")
def tiles():
    return np.concatenate([synth.tiles_u8(3, seed=21, n_slides=2), jpeg_synth.degenerate_tiles(), saturated_tiles()])


@pytest.fixture(scope="module")
def matrix(tiles):
    """(label, bytes, libjpeg-turbo IFAST + replicated pixels): every quality x sampling x restart setting on every
    tile, and the 16-bit-table tiles"""
    out = []
    for q, ss, rs in itertools.product(QUALITIES, SAMPLINGS, RESTARTS):
        for i, t in enumerate(tiles):
            b = jpeg_synth.jpeg_encode(t, q, ss, **rs)
            out.append((f"q{q} {ss} {rs} tile {i}", b, pil_decode_fast(b)))
    for ss, (i, restart) in itertools.product(SAMPLINGS, ((0, None), (4, 2), (9, None))):
        b = dqt16_encode(tiles[i], ss, restart)
        out.append((f"16-bit DQT {ss} restart {restart} tile {i}", b, pil_decode_fast(b)))
    return out


def _first_mismatch(got, want, labels):
    bad = np.flatnonzero((got != want).reshape(len(got), -1).any(1))
    if not bad.size:
        return None
    lines = [f"{bad.size} of {len(got)} tiles differ"]
    for t in bad[:5]:
        y, x, c = np.argwhere(got[t] != want[t])[0]
        lines.append(f"  {labels[t]}: {int((got[t] != want[t]).sum())} values differ; first at pixel ({y}, {x}) "
                     f"component {c}: got {got[t][y, x]} want {want[t][y, x]}")
    return "\n".join(lines)


def test_ifast_replicated_matrix_equals_libjpeg_turbo(matrix, ctx):
    labels, files, want = zip(*matrix)
    got = jpeg.decode(JpegBatch.from_bytes(files, **FAST), ctx=ctx)       # every encoding mixed in one batch
    msg = _first_mismatch(got, np.stack(want), labels)
    assert msg is None, msg
    # "" is INTEGER_FAST
    got = jpeg.decode(JpegBatch.from_bytes(files, dct_method="", fancy_upscaling=False), ctx=ctx)
    assert _first_mismatch(got, np.stack(want), labels) is None


def test_explicit_default_options_equal_the_default_call(matrix, ctx):
    files = [b for _, b, _ in matrix]
    want = jpeg.decode(JpegBatch.from_bytes(files), ctx=ctx)
    got = jpeg.decode(JpegBatch.from_bytes(files, dct_method="INTEGER_ACCURATE", fancy_upscaling=True), ctx=ctx)
    np.testing.assert_array_equal(got, want)
    sub = [files[i] for i in range(0, len(files), 97)]
    np.testing.assert_array_equal(jpeg.decode(JpegBatch.from_bytes(sub), ctx=ctx),
                                  np.stack([jpeg_synth.pil_decode(b) for b in sub]))


@pytest.mark.parametrize("dct_method,fancy", [("INTEGER_FAST", True), ("INTEGER_ACCURATE", False)])
def test_other_combinations_equal_the_restatement(tiles, ctx, dct_method, fancy):
    """IFAST + fancy (TensorFlow's default) and ISLOW + replicated, every sampling, with and without restarts"""
    files = [jpeg_synth.jpeg_encode(tiles[i], q, ss, **rs)
             for ss in SAMPLINGS
             for i, q, rs in ((0, 90, {}), (6, 50, {"restart_rows": 1}), (9, 95, {"restart_blocks": 7}))]
    got = jpeg.decode(JpegBatch.from_bytes(files, dct_method=dct_method, fancy_upscaling=fancy), ctx=ctx)
    want = np.stack([ref_decode(b, dct_method, fancy) for b in files])
    assert _first_mismatch(got, want, [f"file {i}" for i in range(len(files))]) is None


@pytest.mark.parametrize("n", [1, 503, 1200])
def test_batch_sizes_host_and_device(matrix, ctx, n):
    import torch
    pick = np.random.default_rng(n).integers(0, len(matrix), n)
    batch = JpegBatch.from_bytes([matrix[i][1] for i in pick], **FAST)
    want = np.stack([matrix[i][2] for i in pick])
    np.testing.assert_array_equal(jpeg.decode(batch, ctx=ctx), want)
    dev = batch.cuda()
    assert dev.options() == FAST
    out = torch.empty((n, 299, 299, 3), dtype=torch.uint8, device="cuda")
    jpeg.decode(dev, ctx=ctx, out=out)
    np.testing.assert_array_equal(out.cpu().numpy(), want)


def test_options_do_not_leak_between_calls(matrix, ctx):
    files = [b for _, b, _ in matrix[::41]]
    islow = np.stack([jpeg_synth.pil_decode(b) for b in files])
    ifast = np.stack([pil_decode_fast(b) for b in files])
    assert (islow != ifast).any()
    for opts, want in ((None, islow), (FAST, ifast), (None, islow), (FAST, ifast), ({}, islow)):
        batch = JpegBatch.from_bytes(files, **opts) if opts is not None else JpegBatch.from_bytes(files)
        np.testing.assert_array_equal(jpeg.decode(batch, ctx=ctx), want)


def _entropy_start(b):
    sos = b.index(b"\xff\xda")
    return sos + 2 + int.from_bytes(b[sos + 2:sos + 4], "big")


def test_corrupt_entropy_data_raises_with_tile_index(tiles, ctx):
    good = [jpeg_synth.jpeg_encode(t, 90) for t in tiles[:3]]
    s = _entropy_start(good[1])
    cut = s + (len(good[1]) - s) // 2
    while good[1][cut - 1] == 0xFF:
        cut -= 1
    truncated = good[1][:cut] + b"\xff\xd9"
    at = _entropy_start(good[2]) + 40
    while good[2][at - 1] == 0xFF:
        at += 1
    invalid = good[2][:at] + b"\xff\x00" * 4 + good[2][at:]
    for fancy in (True, False):
        opts = dict(dct_method="INTEGER_FAST", fancy_upscaling=fancy)
        with pytest.raises(ValueError, match=r"JPEG tile 1: entropy-coded data truncated"):
            jpeg.decode(JpegBatch.from_bytes([good[0], truncated, good[2]], **opts), ctx=ctx)
        with pytest.raises(ValueError, match=r"JPEG tile 2: invalid Huffman code"):
            jpeg.decode(JpegBatch.from_bytes([good[0], good[1], invalid], **opts), ctx=ctx)
    np.testing.assert_array_equal(jpeg.decode(JpegBatch.from_bytes(good, **FAST), ctx=ctx),
                                  np.stack([pil_decode_fast(b) for b in good]))


@pytest.fixture(scope="module")
def weights():
    from biscuit_b200.weights import random_init
    return random_init(seed=3)


def test_unknown_flag_bits_are_rejected(tiles, weights, ctx):
    lib = ctx.lib
    batch = JpegBatch.from_bytes([jpeg_synth.jpeg_encode(tiles[0], 90)])
    out = np.zeros((1, 299, 299, 3), np.uint8)
    launches = ctx.launches
    for flags in (4, 1 << 30, -1):
        rc = lib.bq_jpeg_decode_ex(ctx.handle, _ffi.ptr(batch.data), _ffi.ptr(batch.offsets), 1, 299, flags,
                                   _ffi.ptr(out), None)
        assert rc == -2                                             # BQ_ERR_ARG
        assert b"unknown decode flag" in lib.bq_last_error(ctx.handle)
    assert ctx.launches == launches
    iface = uq.UncertaintyInterface(weights, max_batch=8, ctx=ctx)
    mean, std = np.zeros((1, 2), np.float32), np.zeros((1, 2), np.float32)
    rc = lib.bq_predict_uq_jpeg_ex(iface.h, _ffi.ptr(batch.data), _ffi.ptr(batch.offsets), 1, 8, 30, C.c_uint64(0),
                                   C.c_uint64(0), None, _ffi.ptr(mean), _ffi.ptr(std), None)
    assert rc == -2 and b"unknown decode flag" in lib.bq_last_error(ctx.handle)
    # the state is usable afterwards, with the options of the next call only
    m, s = iface.predict(JpegBatch.from_bytes([batch.tile(0)], **FAST), T=30, seed=1)
    m_ref, s_ref = iface.predict(pil_decode_fast(batch.tile(0))[None], T=30, seed=1)
    np.testing.assert_array_equal(m, m_ref)
    np.testing.assert_array_equal(s, s_ref)
    iface.close()


@pytest.mark.parametrize("max_batch", [8, uq.BENCH_MICRO_BATCH])
@pytest.mark.parametrize("normalizer", [None, "reinhard_fast"])
def test_predict_ifast_equals_predict_uint8(matrix, weights, ctx, max_batch, normalizer):
    rng = np.random.default_rng(max_batch + 1)
    n = 37 if max_batch == 8 else 700
    files = [matrix[i][1] for i in rng.integers(0, len(matrix), n)]
    iface = uq.UncertaintyInterface(weights, max_batch=max_batch, ctx=ctx, normalizer=normalizer)
    refs = {}
    for method in ("INTEGER_FAST", "INTEGER_ACCURATE"):
        batch = JpegBatch.from_bytes(files, dct_method=method)
        refs[method] = (batch, iface.predict(jpeg.decode(batch, ctx=ctx), T=30, seed=5, tile_index_base=11))
    assert not np.array_equal(refs["INTEGER_FAST"][1][0], refs["INTEGER_ACCURATE"][1][0])
    for method in ("INTEGER_FAST", "INTEGER_ACCURATE", "INTEGER_FAST"):          # alternating on one interface
        batch, (m_ref, s_ref) = refs[method]
        for b in (batch, batch.cuda()):
            m, s = iface.predict(b, T=30, seed=5, tile_index_base=11)
            np.testing.assert_array_equal(m, m_ref, err_msg=method)
            np.testing.assert_array_equal(s, s_ref, err_msg=method)
    iface.close()


def test_predict_tfrecords_ifast_equals_predict_table(tiles, weights, ctx, tmp_path):
    paths, all_files, all_slides, all_locs = [], [], [], []
    k = 0
    for f, (slide, count) in enumerate([("slide A", 5), ("slide B", 4), ("slide A", 6)]):
        files = [jpeg_synth.jpeg_encode(tiles[(k + j) % len(tiles)], 75 + 5 * f, SAMPLINGS[f]) for j in range(count)]
        locs = [(100 * (k + j), 7 * (k + j)) for j in range(count)]
        k += count
        p = tmp_path / f"{f}.tfrecords"
        jpeg_synth.write_tfrecord(p, files, [slide] * count, locs)
        paths.append(p)
        all_files += files
        all_slides += [slide] * count
        all_locs += locs
    iface = uq.UncertaintyInterface(weights, max_batch=8, ctx=ctx)
    labels = {"slide A": 0, "slide B": 1}
    df = uq.predict_tfrecords(iface, paths, y_true=labels, T=30, seed=2, dct_method="INTEGER_FAST")
    pixels = np.stack([ref_decode(b, "INTEGER_FAST") for b in all_files])
    ref = uq.predict_table(iface, pixels, all_slides, y_true=[labels[s] for s in all_slides], T=30, seed=2)
    for col in ref.columns:
        np.testing.assert_array_equal(df[col].to_numpy(), ref[col].to_numpy(), err_msg=col)
    assert df["loc_x"].tolist() == [x for x, _ in all_locs] and df["loc_y"].tolist() == [y for _, y in all_locs]
    default = uq.predict_tfrecords(iface, paths, y_true=labels, T=30, seed=2)
    assert not np.array_equal(default["uncertainty"].to_numpy(), df["uncertainty"].to_numpy())
    threshold.apply(df.drop(columns=["loc_x", "loc_y"]), 0.5, 0.5)
    iface.close()
