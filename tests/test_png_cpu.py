"""CPU tier of the PNG input: the test generators are pinned (every valid file round-trips through Pillow, every
hand-made stream is accepted or rejected as zlib.decompress does), the host chunk parse (bq_png_inspect) accepts every
encoding of the matrix and rejects each header case with its own message, and tfrecord.read picks the batch class by
the images' format."""
import struct
import zlib

import numpy as np
import pytest

from biscuit_b200 import png, tfrecord
from biscuit_b200.jpeg import JpegBatch
from biscuit_b200.png import PngBatch
from oracle import jpeg_synth, png_synth, synth

PX = synth.TILE_PX
ROW = 1 + 3 * PX


@pytest.fixture(scope="module")
def tile():
    return synth.tiles_u8(1, seed=4)[0]


def test_every_encoding_round_trips_through_pillow(tile):
    tiles = [tile, jpeg_synth.degenerate_tiles()[3], png_synth.distance_tile()]
    for t in tiles:
        for label, kw in png_synth.encodings():
            np.testing.assert_array_equal(png_synth.pil_decode(png_synth.png_encode(t, **kw)), t, err_msg=label)
        for k in png_synth.PIL_LEVELS:
            np.testing.assert_array_equal(png_synth.pil_decode(png_synth.pil_encode(t, k)), t)


def test_distance_tile_has_matches_near_the_window_limit():
    t = png_synth.distance_tile()
    raw = png_synth.filter_rows(t, [0] * PX)
    assert 36 * ROW == 32328
    assert raw[36 * ROW:] == raw[:-36 * ROW]       # every row after the 36th repeats the one 32,328 bytes back
    z = zlib.compress(raw, 9)
    assert len(z) < len(raw) // 4                  # so the encoder did use those distances


def test_crafted_streams_follow_zlib(tile):
    raw = png_synth.filter_rows(tile, np.arange(PX) % 5)
    cases = png_synth.crafted_streams(raw, ROW)
    for name, (z, status, got) in cases.items():
        # zlib rejects every stream whose error is in the DEFLATE data or its trailer; it accepts the wrong-size and
        # bad-filter streams (PNG-level errors), and the valid ones
        zlib_ok = status in (None, "wrong decompressed size", "bad filter type")
        assert (got is not None) == zlib_ok, name
        f = png_synth.assemble(PX, PX, z)
        try:
            pil = png_synth.pil_decode(f)
        except Exception:
            pil = None
        if status is None:
            assert pil is not None, name           # every file the GPU accepts, Pillow accepts
        elif status not in ("wrong decompressed size", "truncated data"):
            assert pil is None, name
    # zlib does not hold a match to the window the header declares (CINFO = 1: 512 bytes) as long as it lies inside
    # the output; the GPU decoder follows it
    z, status, got = cases["distance beyond the declared window"]
    assert z[0] >> 4 == 1 and status is None and got is not None
    # the two documented deviations: Pillow stops once the image is full
    assert png_synth.pil_decode(png_synth.assemble(PX, PX, cases["three bytes long"][0])).shape == (PX, PX, 3)
    assert png_synth.pil_decode(png_synth.assemble(PX, PX, cases["no Adler-32"][0])).shape == (PX, PX, 3)


def test_inspect_accepts_every_encoding_of_the_matrix(tile):
    files = [png_synth.png_encode(tile, **kw) for _, kw in png_synth.encodings()]
    files += [png_synth.pil_encode(tile, k) for k in png_synth.PIL_LEVELS]
    st = png.inspect(PngBatch.from_bytes(files))
    assert st.tolist() == [0] * len(files)


def _with_zlib_header(good, cmf, flg):
    i = good.index(b"IDAT") + 4
    return good[:i] + bytes([cmf, flg]) + good[i + 2:]


def test_inspect_rejections_each_with_its_own_message(tile):
    good = png_synth.png_encode(tile, filters="random", idat_size=8192)
    sig_ihdr = png_synth.SIGNATURE + png_synth.ihdr(PX, PX)
    z = zlib.compress(b"\0")
    bad_crc = bytearray(good)
    bad_crc[8 + 8 + 3] ^= 1                       # a byte of IHDR's width
    cases = {
        "not a PNG": jpeg_synth.jpeg_encode(tile, 90),
        "truncated header": good[:40],
        "bad chunk CRC": bytes(bad_crc),
        "bad IHDR": png_synth.SIGNATURE + png_synth.chunk(b"IHDR", struct.pack(">IIBBBBBB", PX, PX, 8, 2, 0, 0, 0, 0))
        + png_synth.chunk(b"IDAT", z),
        "size": png_synth.png_encode(np.zeros((300, 300, 3), np.uint8)),
        "bit depth": png_synth.assemble(PX, PX, z, header=png_synth.ihdr(PX, PX, depth=16)),
        "grayscale": png_synth.pil_encode(tile, mode="L"),
        "interlaced": png_synth.assemble(PX, PX, z, header=png_synth.ihdr(PX, PX, interlace=1)),
        "unknown critical chunk": png_synth.assemble(PX, PX, z, before=[png_synth.chunk(b"ABCD", b"xyz")]),
        "no IDAT": sig_ihdr + png_synth.chunk(b"IEND", b""),
        "bad zlib header": _with_zlib_header(good, 0x88, 0x1C),          # CINFO 8: a 64 KB window
        "preset dictionary": _with_zlib_header(good, 0x78, 0xBB),        # FDICT set, FCHECK valid
    }
    assert (0x88 << 8 | 0x1C) % 31 == 0 and (0x78 << 8 | 0xBB) % 31 == 0
    batch = PngBatch.from_bytes([good] + list(cases.values()))
    st = png.inspect(batch)
    assert st[0] == 0
    msgs = [png.status_message(s) for s in st[1:]]
    assert all(s != 0 for s in st[1:])
    assert len(set(msgs)) == len(msgs), msgs
    for (key, _), m in zip(cases.items(), msgs):
        assert key.lower() in m.lower(), (key, m)
    # every colour type other than RGB has the same message
    for mode in ("P", "RGBA", "LA"):
        s = png.inspect(PngBatch.from_bytes([png_synth.pil_encode(tile, mode=mode)]))[0]
        assert "colour type" in png.status_message(s), mode
    with pytest.raises(ValueError, match=r"PNG tile 1: not a PNG"):
        png.check(batch)


def test_ancillary_chunks_and_plte_are_skipped_and_checked(tile):
    z = zlib.compress(png_synth.filter_rows(tile, [0] * PX))
    plte = png_synth.chunk(b"PLTE", bytes(range(48)))
    ok = png_synth.assemble(PX, PX, z, idat_size=1, before=png_synth.ancillary(3000) + [plte])
    bad = bytearray(png_synth.assemble(PX, PX, z, before=png_synth.ancillary()))
    bad[bad.index(b"pHYs") + 5] ^= 1               # ancillary chunks before IDAT must pass their CRC too
    st = png.inspect(PngBatch.from_bytes([ok, bytes(bad)]))
    assert st[0] == 0 and "CRC" in png.status_message(st[1])


def test_png_batch_is_its_own_class():
    b = PngBatch.from_bytes([b"\x89PNG", b"xy"])
    assert type(b) is PngBatch and not isinstance(b, JpegBatch) and len(b) == 2 and b.tile(1) == b"xy"
    assert type(JpegBatch.from_bytes([b"ab"])) is JpegBatch


def test_tfrecord_read_picks_the_batch_class(tile, tmp_path):
    pngs = [png_synth.pil_encode(t) for t in synth.tiles_u8(3, seed=8)]
    jpegs = [jpeg_synth.jpeg_encode(t, 90) for t in synth.tiles_u8(2, seed=8)]
    pa, pb, pc = tmp_path / "a.tfrecords", tmp_path / "b.tfrecords", tmp_path / "c.tfrecords"
    jpeg_synth.write_tfrecord(pa, pngs, ["s"] * 3, [(0, 1)] * 3)
    jpeg_synth.write_tfrecord(pb, jpegs, ["t"] * 2)
    jpeg_synth.write_tfrecord(pc, pngs[:1] + jpegs[:1], ["u"] * 2)
    batch, slides, lx, ly = tfrecord.read([pa, pa])
    assert type(batch) is PngBatch and len(batch) == 6 and [batch.tile(i) for i in range(3)] == pngs
    assert type(tfrecord.read(pb)[0]) is JpegBatch
    garbage = tmp_path / "g.tfrecords"
    jpeg_synth.write_tfrecord(garbage, [b"neither"] + jpegs, ["v"] * 3)
    assert type(tfrecord.read(garbage)[0]) is JpegBatch     # not PNG: the JPEG decoder reports it
    with pytest.raises(ValueError, match=r"b\.tfrecords record 0: image is not PNG"):
        tfrecord.read([pa, pb])
    with pytest.raises(ValueError, match=r"c\.tfrecords record 1: image is not PNG"):
        tfrecord.read(pc)
    with pytest.raises(ValueError, match=r"a\.tfrecords record 0: image is PNG"):
        tfrecord.read([pb, pa])
