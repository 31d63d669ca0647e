"""GPU tier of the compressed-tile driver shared by JPEG and PNG (csrc/encoded.cu), each case run for both formats:
headers that run past the head fetched from device memory, a header rejected from device-resident bytes, an empty
batch, and both formats alternating on one context and one `UncertaintyInterface` at batch sizes that grow the
scratch."""
import numpy as np
import pytest

from biscuit_b200 import jpeg, png, uq
from biscuit_b200.jpeg import JpegBatch
from biscuit_b200.png import PngBatch
from oracle import jpeg_synth, png_synth, synth

pytestmark = pytest.mark.gpu

PX = synth.TILE_PX
FORMATS = {"jpeg": (jpeg, JpegBatch, jpeg_synth.pil_decode), "png": (png, PngBatch, png_synth.pil_decode)}


@pytest.fixture(scope="module")
def tiles():
    return np.concatenate([synth.tiles_u8(4, seed=33, n_slides=2), jpeg_synth.degenerate_tiles()[:2]])


@pytest.fixture(scope="module")
def files(tiles):
    """a few encodings of every tile per format: (bytes, Pillow pixels)"""
    out = {"jpeg": [], "png": []}
    for t in tiles:
        for q, ss in ((75, "4:2:0"), (95, "4:4:4"), (90, "4:2:2")):
            out["jpeg"].append(jpeg_synth.jpeg_encode(t, q, ss))
        for level in (1, 6):
            out["png"].append(png_synth.pil_encode(t, level))
    return {fmt: [(b, FORMATS[fmt][2](b)) for b in bs] for fmt, bs in out.items()}


def _long_headers(fmt, tile):
    """a file whose headers run past the head the driver fetches per device-resident tile (2 KB JPEG, 1 KB PNG)"""
    if fmt == "jpeg":
        b = jpeg_synth.jpeg_encode(tile, 90)
        com = bytes(np.random.default_rng(1).integers(0, 256, 3000, dtype=np.uint8)).replace(b"\xff", b"\x00")
        return b[:2] + b"\xff\xfe" + (len(com) + 2).to_bytes(2, "big") + com + b[2:]
    return png_synth.png_encode(tile, filters=4, before=png_synth.ancillary(iccp_bytes=3000))


def _plain(fmt, tile):
    return jpeg_synth.jpeg_encode(tile, 90) if fmt == "jpeg" else png_synth.pil_encode(tile)


def _rejected(fmt, tile):
    if fmt == "jpeg":
        return jpeg_synth.jpeg_encode(tile, 90, progressive=True), r"JPEG tile 1: progressive"
    return png_synth.pil_encode(tile, mode="L"), r"PNG tile 1: colour type"


@pytest.mark.parametrize("fmt", FORMATS)
def test_headers_past_the_head_from_device(fmt, tiles, ctx):
    mod, Batch, pil = FORMATS[fmt]
    long = _long_headers(fmt, tiles[0])
    assert long.index(b"\xff\xda" if fmt == "jpeg" else b"IDAT") > 3000
    files = [_plain(fmt, tiles[1]), long]
    want = np.stack([pil(b) for b in files])
    np.testing.assert_array_equal(mod.decode(Batch.from_bytes(files).cuda(), ctx=ctx), want)


@pytest.mark.parametrize("fmt", FORMATS)
def test_header_rejected_from_device_bytes(fmt, tiles, ctx):
    mod, Batch, _ = FORMATS[fmt]
    good = _plain(fmt, tiles[0])
    bad, pattern = _rejected(fmt, tiles[0])
    batch = Batch.from_bytes([good, bad])
    with pytest.raises(ValueError, match=pattern) as host:
        mod.decode(batch, ctx=ctx)
    dev = batch.cuda()
    launches = ctx.launches
    with pytest.raises(ValueError, match=pattern) as device:
        mod.decode(dev, ctx=ctx)
    assert str(device.value) == str(host.value)
    assert ctx.launches == launches + 1            # the head gather only


@pytest.fixture(scope="module")
def weights():
    from biscuit_b200.weights import random_init
    return random_init(seed=3)


@pytest.mark.parametrize("fmt", FORMATS)
def test_empty_batch(fmt, weights, ctx):
    mod, Batch, _ = FORMATS[fmt]
    iface = uq.UncertaintyInterface(weights, max_batch=8, ctx=ctx)
    nc = iface.config.n_classes
    for batch in (Batch.from_bytes([]), Batch.from_bytes([]).cuda()):
        assert mod.decode(batch, ctx=ctx).shape == (0, PX, PX, 3)
        m, s = iface.predict(batch, T=30, seed=5)
        assert m.shape == (0, nc) and s.shape == (0, nc)
    iface.close()


def test_formats_alternate_on_one_context_and_interface(files, weights, ctx):
    iface = uq.UncertaintyInterface(weights, max_batch=uq.BENCH_MICRO_BATCH, ctx=ctx)
    rng = np.random.default_rng(7)
    for k, (fmt, n, on_device) in enumerate((("jpeg", 37, False), ("png", 700, False), ("jpeg", 700, True),
                                             ("png", 37, False))):
        mod, Batch, _ = FORMATS[fmt]
        pick = rng.integers(0, len(files[fmt]), n)
        batch = Batch.from_bytes([files[fmt][i][0] for i in pick])
        pixels = np.stack([files[fmt][i][1] for i in pick])
        if on_device:
            batch = batch.cuda()
        m_ref, s_ref = iface.predict(pixels, T=30, seed=5, tile_index_base=k)
        m, s = iface.predict(batch, T=30, seed=5, tile_index_base=k)
        np.testing.assert_array_equal(m, m_ref, err_msg=f"{fmt} n={n}")
        np.testing.assert_array_equal(s, s_ref, err_msg=f"{fmt} n={n}")
        # the other format's decode on the same context in between, then this one's
        other = "png" if fmt == "jpeg" else "jpeg"
        omod, OBatch, _ = FORMATS[other]
        opick = rng.integers(0, len(files[other]), n)
        np.testing.assert_array_equal(omod.decode(OBatch.from_bytes([files[other][i][0] for i in opick]), ctx=ctx),
                                      np.stack([files[other][i][1] for i in opick]), err_msg=f"{other} n={n}")
        np.testing.assert_array_equal(mod.decode(batch, ctx=ctx), pixels, err_msg=f"{fmt} n={n}")
    iface.close()
