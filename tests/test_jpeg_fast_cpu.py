"""CPU tier of TensorFlow's decode_jpeg options (dct_method, fancy_upscaling): the numpy restatement of libjpeg-turbo's
IFAST IDCT and replicated chroma (tests/jpeg_fast_ref.py) pinned bit for bit to libjpeg-turbo through Pillow's draft
decode, and the option values JpegBatch / tfrecord.read accept."""
import itertools

import numpy as np
import pytest

from biscuit_b200 import _ffi, tfrecord
from biscuit_b200.jpeg import JpegBatch
from biscuit_b200.png import PngBatch
from jpeg_fast_ref import DCT_METHODS, decode, dqt16_encode, ifast_multipliers, pil_decode_fast, saturated_tiles
from oracle import jpeg_ref, jpeg_synth, png_synth, synth

QUALITIES = (1, 10, 25, 50, 75, 90, 95, 100)
SAMPLINGS = ("4:4:4", "4:2:2", "4:2:0")
RESTARTS = ({}, {"restart_blocks": 7}, {"restart_rows": 1})


def tile_pool():
    return np.concatenate([synth.tiles_u8(2, seed=31, n_slides=2), jpeg_synth.degenerate_tiles(), saturated_tiles()])


@pytest.mark.parametrize("subsampling", SAMPLINGS)
def test_ifast_replicated_matches_libjpeg_turbo(subsampling):
    """every quality x restart setting, two tiles per cell, rotating through synthetic, degenerate and saturated tiles"""
    pool = tile_pool()
    k = SAMPLINGS.index(subsampling)
    for qi, q in enumerate(QUALITIES):
        for j in range(2):
            rs = RESTARTS[(qi + j + k) % len(RESTARTS)]
            ti = (2 * qi + j + 3 * k) % len(pool)
            b = jpeg_synth.jpeg_encode(pool[ti], q, subsampling, **rs)
            np.testing.assert_array_equal(decode(b, "INTEGER_FAST", fancy_upscaling=False), pil_decode_fast(b),
                                          err_msg=f"q{q} {subsampling} {rs} tile {ti}")


@pytest.mark.parametrize("subsampling", SAMPLINGS)
def test_ifast_replicated_matches_libjpeg_turbo_16bit_tables(subsampling):
    pool = tile_pool()
    lum = np.linspace(200, 20063, 64).astype(np.int64)
    assert (((lum[::-1] * 16384 + 2048) >> 12) > 32767).any()      # the multiplier's int16 cast matters here
    for ti, restart in ((0, None), (6, 3), (8, None)):
        b = dqt16_encode(pool[ti], subsampling, restart)
        dqt = b.index(b"\xff\xdb")
        assert b[dqt + 4] >> 4 == 1, "Pillow wrote 8-bit tables"
        np.testing.assert_array_equal(decode(b, "", fancy_upscaling=False), pil_decode_fast(b),
                                      err_msg=f"16-bit DQT {subsampling} tile {ti} restart {restart}")


def test_draft_decode_is_not_the_default_decode():
    """the pin above means something only while Pillow's draft route really is a different decoder"""
    t = synth.tiles_u8(1, seed=6)[0]
    for q, ss in ((100, "4:4:4"), (95, "4:2:0")):
        b = jpeg_synth.jpeg_encode(t, q, ss)
        fast, default = pil_decode_fast(b), jpeg_synth.pil_decode(b)
        assert (fast != default).mean() > 0.25, (q, ss)


def test_default_options_are_the_default_decode():
    pool = tile_pool()
    for q, ss, ti in ((50, "4:4:4", 0), (90, "4:2:2", 5), (100, "4:2:0", 7)):
        b = jpeg_synth.jpeg_encode(pool[ti], q, ss)
        want = jpeg_ref.decode(b)
        np.testing.assert_array_equal(decode(b), want)
        np.testing.assert_array_equal(decode(b, "INTEGER_ACCURATE", fancy_upscaling=True), want)
        if ss == "4:4:4":      # upsampling has nothing to do
            np.testing.assert_array_equal(decode(b, "INTEGER_ACCURATE", fancy_upscaling=False), want)


def test_ifast_multipliers_follow_jddctmgr():
    q = np.arange(64) * 1000 + 1
    s = np.array([1.0] + [np.sqrt(2) * np.cos(k * np.pi / 16) for k in range(1, 8)])
    aan = np.round(16384 * np.outer(s, s)).astype(np.int64).ravel()
    want = (((q * aan + 2048) >> 12) + 32768) % 65536 - 32768
    np.testing.assert_array_equal(ifast_multipliers(q), want)
    assert ifast_multipliers(np.full(64, 1))[0] == 4                 # 1 * 16384 / 4096


# ------------------------------------------------------------------------------------------------------------------
# the option values
# ------------------------------------------------------------------------------------------------------------------
def test_dct_method_values_and_flags():
    b = [jpeg_synth.jpeg_encode(synth.tiles_u8(1, seed=1)[0], 75)]
    assert JpegBatch.from_bytes(b).flags == 0
    assert JpegBatch.from_bytes(b, dct_method="INTEGER_ACCURATE").flags == 0
    assert JpegBatch.from_bytes(b, dct_method="INTEGER_FAST").flags == _ffi.BQ_JPEG_IDCT_IFAST
    assert JpegBatch.from_bytes(b, dct_method="").flags == _ffi.BQ_JPEG_IDCT_IFAST          # TensorFlow: "" = FAST
    assert JpegBatch.from_bytes(b, fancy_upscaling=False).flags == _ffi.BQ_JPEG_REPLICATE_CHROMA
    both = JpegBatch.from_bytes(b, dct_method="", fancy_upscaling=False)
    assert both.flags == _ffi.BQ_JPEG_IDCT_IFAST | _ffi.BQ_JPEG_REPLICATE_CHROMA
    assert both.options() == dict(dct_method="", fancy_upscaling=False)
    assert JpegBatch(both.data, both.offsets, **both.options()).flags == both.flags
    for bad in ("INTEGER_FLOAT", "integer_fast", "FAST", None, 1):
        with pytest.raises(ValueError, match="dct_method"):
            JpegBatch.from_bytes(b, dct_method=bad)
    with pytest.raises(ValueError, match="fancy_upscaling"):
        JpegBatch.from_bytes(b, fancy_upscaling="False")
    with pytest.raises(ValueError, match="dct_method"):
        decode(b[0], "INTEGER_FLOAT")
    assert sorted(DCT_METHODS) == ["", "INTEGER_ACCURATE", "INTEGER_FAST"]


def test_tfrecord_read_passes_the_options_to_jpeg_only(tmp_path):
    tiles = synth.tiles_u8(2, seed=2)
    p = tmp_path / "jpeg.tfrecords"
    jpeg_synth.write_tfrecord(p, [jpeg_synth.jpeg_encode(t, 80) for t in tiles], ["a", "b"])
    batch = tfrecord.read(p)[0]
    assert isinstance(batch, JpegBatch) and batch.flags == 0
    for method, fancy in itertools.product(("INTEGER_FAST", "", "INTEGER_ACCURATE"), (True, False)):
        batch = tfrecord.read(p, dct_method=method, fancy_upscaling=fancy)[0]
        assert (batch.dct_method, batch.fancy_upscaling) == (method, fancy)
    with pytest.raises(ValueError, match="dct_method"):
        tfrecord.read(p, dct_method="INTEGER_FLOAT")
    q = tmp_path / "png.tfrecords"
    jpeg_synth.write_tfrecord(q, [png_synth.png_encode(t) for t in tiles], ["a", "b"])
    batch = tfrecord.read(q, dct_method="INTEGER_FAST", fancy_upscaling=False)[0]
    assert isinstance(batch, PngBatch) and batch.flags is None
