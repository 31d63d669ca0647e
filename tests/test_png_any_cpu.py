"""CPU tier of the PNG decode option `convert_rgb`: the test reference decoder (tests/png_any_ref.py) equals Pillow's
`convert("RGB")` on every colour type, bit depth, interlace and filter the writer makes and on Pillow's own encodings,
with 16-bit grayscale pinned as the one documented difference; the host chunk parse (bq_png_inspect_ex) accepts the
whole matrix under the option and still rejects it without; each new rejection has its own message; the option
travels with the batch and through tfrecord.read."""
import io
import struct

import numpy as np
import pytest

import png_any_ref as R
from biscuit_b200 import _ffi, png, tfrecord
from biscuit_b200.png import PngBatch
from oracle import jpeg_synth, png_synth, synth

PX = synth.TILE_PX
BQ_ERR_ARG = -2       # include/biscuit_b200.h


def _pil(b):
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))


@pytest.mark.filterwarnings("ignore:Palette images with Transparency")
@pytest.mark.parametrize("interlace", [0, 1])
@pytest.mark.parametrize("colour,depth", R.COMBOS)
def test_reference_equals_pillow(colour, depth, interlace):
    cases = [(61, f, s) for s, f in enumerate(R.FILTER_MODES)] + [(PX, "random", 9), (1, 0, 1), (9, "random", 2)]
    for px, filters, seed in cases:
        s = R.random_samples(px, colour, depth, seed)
        pal = R.random_palette(min(256, (1 << depth) - 1 or 1), seed) if colour == 3 else None
        trns = {0: struct.pack(">H", 1), 2: struct.pack(">HHH", 1, 2, 3), 3: b"\x00\x80"}.get(colour)
        b = R.encode(s, colour, depth, interlace, filters, pal, seed, trns=trns)
        want = R.to_rgb(s, colour, depth, pal)
        msg = f"{R.label(colour, depth, interlace)} px {px} filters {filters}"
        np.testing.assert_array_equal(R.decode(b), want, err_msg=msg)
        if (colour, depth) == (0, 16):
            # Pillow opens 16-bit gray as "I;16" and clips it to 255; the decoder takes the high byte
            np.testing.assert_array_equal(_pil(b), np.repeat(np.minimum(s, 255), 3, 2).astype(np.uint8), err_msg=msg)
            assert px == 1 or not np.array_equal(_pil(b), want)
        else:
            np.testing.assert_array_equal(_pil(b), want, err_msg=msg)


@pytest.mark.parametrize("mode", ["L", "LA", "RGBA", "P", "1", "RGB"])
def test_reference_decodes_pillow_encodings(mode):
    from PIL import Image
    tile = synth.tiles_u8(1, seed=8)[0]
    img = Image.fromarray(tile).convert(mode) if mode != "RGBA" else Image.fromarray(
        np.dstack([tile, tile[..., :1]]), "RGBA")
    for kw in ({}, {"optimize": True}):
        bio = io.BytesIO()
        img.save(bio, "PNG", **kw)
        b = bio.getvalue()
        np.testing.assert_array_equal(R.decode(b), _pil(b), err_msg=f"{mode} {kw}")


def test_palette_index_past_plte_is_black():
    s = np.arange(16, dtype=np.uint16).reshape(4, 4, 1)
    pal = bytes(range(1, 16)) + b"\x09\x08\x07"         # 6 entries: indices 6-15 are out of range
    b = R.encode(s, 3, 4, 0, 0, pal)
    got = R.decode(b)
    assert (got.reshape(-1, 3)[6:] == 0).all()
    np.testing.assert_array_equal(got.reshape(-1, 3)[:6], np.frombuffer(pal, np.uint8).reshape(6, 3))
    np.testing.assert_array_equal(_pil(b), got)


@pytest.fixture(scope="module")
def matrix_files():
    return [(R.label(c, d, il), R.make(PX, c, d, il, seed=c * 17 + d)[0]) for c, d in R.COMBOS for il in (0, 1)]


def test_inspect_ex_accepts_the_matrix_only_under_the_option(matrix_files):
    labels, files = zip(*matrix_files)
    on = png.inspect(PngBatch.from_bytes(files, convert_rgb=True))
    assert (on == 0).all(), [l for l, s in zip(labels, on) if s]
    off = png.inspect(PngBatch.from_bytes(files))
    for l, f, s in zip(labels, files, off):
        if l == "RGB 8-bit":
            assert s == 0
        else:
            assert s != 0, l
    np.testing.assert_array_equal(off, png.inspect(PngBatch.from_bytes(files, convert_rgb=False)))
    # the old entry point and the option-less batch give the same statuses
    lib = _ffi.load_library()
    batch = PngBatch.from_bytes(files)
    st = np.zeros(len(files), np.int32)
    assert lib.bq_png_inspect(_ffi.ptr(batch.data), _ffi.ptr(batch.offsets), len(files), PX, _ffi.ptr(st)) == 0
    np.testing.assert_array_equal(st, off)


def test_inspect_ex_rejects_unknown_flags(matrix_files):
    batch = PngBatch.from_bytes([matrix_files[0][1]])
    st = np.zeros(1, np.int32)
    lib = _ffi.load_library()
    assert lib.bq_png_inspect_ex(_ffi.ptr(batch.data), _ffi.ptr(batch.offsets), 1, PX, 2, _ffi.ptr(st)) == BQ_ERR_ARG


def _with_header(colour, depth, plte=None, interlace=0):
    s = R.random_samples(8, 0, 8)                       # any stream: only the header is parsed
    z = png_synth.zlib_stream(R.filter_rows(R.pack(s, 8), [0] * 8, 1))
    before = [png_synth.chunk(b"PLTE", plte)] if plte is not None else []
    return png_synth.assemble(8, 8, z, before=before, header=png_synth.ihdr(8, 8, depth, colour, interlace))


def test_new_rejections_each_with_its_own_message():
    cases = {
        "gray 3-bit": (_with_header(0, 3), "bad IHDR"),
        "RGB 4-bit": (_with_header(2, 4), "bad IHDR"),
        "palette 16-bit": (_with_header(3, 16, b"\0\0\0"), "bad IHDR"),
        "gray+alpha 4-bit": (_with_header(4, 4), "bad IHDR"),
        "RGBA 1-bit": (_with_header(6, 1), "bad IHDR"),
        "colour type 5": (_with_header(5, 8), "bad IHDR"),
        "palette, no PLTE": (_with_header(3, 8), "palette image without a PLTE chunk"),
        "PLTE length 0": (_with_header(3, 8, b""), r"bad PLTE \(length 0"),
        "PLTE length 4": (_with_header(3, 8, b"\0" * 4), r"bad PLTE \(length 0, not a multiple of 3"),
        "PLTE 257 entries": (_with_header(3, 8, b"\0" * 771), r"bad PLTE .*more than 256 entries"),
    }
    messages = set()
    for name, (f, msg) in cases.items():
        batch = PngBatch.from_bytes([_with_header(2, 8), f], convert_rgb=True)
        with pytest.raises(ValueError, match=rf"PNG tile 1: {msg}"):
            png.check(batch, 8)
        messages.add(png.status_message(int(png.inspect(batch, 8)[1])))
    assert len(messages) == 3
    assert png.status_message(13) != png.status_message(14) and "unknown" not in png.status_message(13)
    # a valid palette image and PLTE in an RGB / gray image are accepted (PLTE skipped there)
    ok = [_with_header(3, 8, b"\1\2\3" * 256), _with_header(2, 8, b"\0" * 6), _with_header(0, 8, b"\0" * 6),
          _with_header(3, 1, b"\1\2\3")]
    assert (png.inspect(PngBatch.from_bytes(ok, convert_rgb=True), 8) == 0).all()
    # a PLTE whose CRC is wrong is still a CRC error, with or without the option
    for colour, opts in ((2, (False, True)), (3, (True,))):
        bad = bytearray(_with_header(colour, 8, b"\1\2\3"))
        bad[8 + 25 + 8] ^= 1
        for opt in opts:
            assert png.inspect(PngBatch.from_bytes([bytes(bad)], convert_rgb=opt), 8)[0] == 3


def test_option_off_keeps_the_old_statuses():
    # the existing rejections without the option: colour type, bit depth, interlace
    st = png.inspect(PngBatch.from_bytes([_with_header(0, 8), _with_header(2, 16), _with_header(2, 8, interlace=1),
                                          _with_header(3, 8)]), 8)
    assert list(st) == [7, 6, 8, 7]


def test_batch_carries_the_option():
    f = [_with_header(2, 8)]
    assert PngBatch.from_bytes(f).flags is None and PngBatch.from_bytes(f).options() == {"convert_rgb": False}
    b = PngBatch.from_bytes(f, convert_rgb=True)
    assert b.flags == _ffi.BQ_PNG_CONVERT_RGB and b.options() == {"convert_rgb": True}
    with pytest.raises(ValueError, match="convert_rgb must be a bool"):
        PngBatch(b.data, b.offsets, convert_rgb="yes")


def test_tfrecord_read_passes_the_option(tmp_path, matrix_files):
    files = [f for _, f in matrix_files[:4]]
    p = tmp_path / "a.tfrecords"
    jpeg_synth.write_tfrecord(p, files, ["s"] * 4, [(i, i) for i in range(4)])
    assert tfrecord.read(p)[0].convert_rgb is False
    batch = tfrecord.read(p, png_convert_rgb=True)[0]
    assert isinstance(batch, PngBatch) and batch.convert_rgb
    assert (png.inspect(batch) == 0).all()
    # ignored for JPEG records
    j = tmp_path / "j.tfrecords"
    tile = synth.tiles_u8(1, seed=1)[0]
    jpeg_synth.write_tfrecord(j, [jpeg_synth.jpeg_encode(tile)], ["s"], [(0, 0)])
    assert tfrecord.read(j, png_convert_rgb=True)[0].FORMAT == "jpeg"
