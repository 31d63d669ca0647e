"""GPU tier of the PNG decode option `convert_rgb`: every colour type x bit depth x interlace x filter mode decodes bit
for bit as the test reference decoder does (tests/png_any_ref.py), at 299 px and at 1 to 9 px (empty Adam7 passes);
8-bit RGB tiles decode to the same bytes with the option as without it; mixed batches over several groups from host
and device bytes; corrupt streams name the tile and leave the others decoded; `predict` and `predict_tfrecords`
with the option equal `predict` / `predict_table` on the reference-decoded tiles."""
import zlib

import numpy as np
import pytest

import png_any_ref as R
from biscuit_b200 import png, uq
from biscuit_b200.png import PngBatch
from oracle import jpeg_synth, png_synth, synth

pytestmark = pytest.mark.gpu

PX = synth.TILE_PX


@pytest.fixture(scope="module")
def matrix():
    """(label, bytes, reference pixels, (width, interlace)) of every colour type x depth x interlace x filter mode"""
    out = []
    for k, (c, d) in enumerate(R.COMBOS):
        for il in (0, 1):
            for j, f in enumerate(R.FILTER_MODES):
                b, _ = R.make(PX, c, d, il, f, seed=100 * k + 10 * il + j)
                out.append((f"{R.label(c, d, il)} filters {f}", b, R.decode(b), (PX, il)))
    return out


def _check(got, entries):
    labels, _, want, meta = zip(*entries)
    msg = R.first_mismatch(got, np.stack(want), labels, meta)
    assert msg is None, msg


def test_full_matrix_bit_exact(matrix, ctx):
    got = png.decode(PngBatch.from_bytes([m[1] for m in matrix], convert_rgb=True), ctx=ctx)
    _check(got, matrix)


@pytest.mark.parametrize("px", range(1, 10))
def test_small_sizes_and_empty_passes(px, ctx):
    entries = []
    for k, (c, d) in enumerate(R.COMBOS):
        for il in (0, 1):
            b, want = R.make(px, c, d, il, "random", seed=7 * k + il + 1000 * px)
            assert np.array_equal(R.decode(b), want)
            entries.append((R.label(c, d, il), b, want, (px, il)))
    batch = PngBatch.from_bytes([e[1] for e in entries], convert_rgb=True)
    _check(png.decode(batch, px, ctx=ctx), entries)
    _check(png.decode(batch.cuda(), px, ctx=ctx), entries)


def test_rgb8_same_bytes_with_and_without_the_option(ctx):
    tiles = np.concatenate([synth.tiles_u8(2, seed=21), jpeg_synth.degenerate_tiles()[:2],
                            png_synth.distance_tile()[None]])
    files = [png_synth.png_encode(t, **kw) for t in tiles for _, kw in png_synth.encodings()]
    files += [png_synth.pil_encode(t, k) for t in tiles for k in png_synth.PIL_LEVELS]
    off = png.decode(PngBatch.from_bytes(files), ctx=ctx)
    on = png.decode(PngBatch.from_bytes(files, convert_rgb=True), ctx=ctx)
    np.testing.assert_array_equal(on, off)
    np.testing.assert_array_equal(on, np.stack([png_synth.pil_decode(b) for b in files]))


@pytest.mark.parametrize("n", [503, 1200])
def test_mixed_batches_host_and_device(matrix, ctx, n):
    import torch
    rng = np.random.default_rng(n)
    rgb8 = [png_synth.pil_encode(t) for t in synth.tiles_u8(3, seed=5)]
    pool = [(m[0], m[1], m[2], m[3]) for m in matrix] + [("Pillow RGB8", b, png_synth.pil_decode(b), (PX, 0))
                                                         for b in rgb8]
    entries = [pool[i] for i in rng.integers(0, len(pool), n)]
    batch = PngBatch.from_bytes([e[1] for e in entries], convert_rgb=True)
    for b in (batch, batch.cuda()):
        assert b.convert_rgb
        _check(png.decode(b, ctx=ctx), entries)
        out = torch.empty((n, PX, PX, 3), dtype=torch.uint8, device="cuda")
        png.decode(b, ctx=ctx, out=out)
        _check(out.cpu().numpy(), entries)


def _corrupt_cases():
    """(name, file, message) of three tiles the kernels must reject"""
    cases = []
    # interlaced RGBA 8-bit, its decompressed stream one byte short
    s = R.random_samples(PX, 6, 8, seed=1)
    raw = R.filtered(s, 6, 8, 1)
    cases.append(("one byte short", R.assemble(PX, PX, 6, 8, 1, zlib.compress(raw[:-1])), "wrong decompressed size"))
    # interlaced gray 4-bit, filter type 5 on the first row of pass 7
    s = R.random_samples(PX, 0, 4, seed=2)
    raw = bytearray(R.filtered(s, 0, 4, 1))
    pass7 = [p for p in R.passes(PX, PX, 1) if p[0] == 6][0]
    at = len(raw) - pass7[6] * R.row_bytes(pass7[5], 0, 4)
    raw[at] = 5
    cases.append(("filter 5 in pass 7", R.assemble(PX, PX, 0, 4, 1, zlib.compress(bytes(raw))), "bad filter type"))
    # RGB 16-bit with a wrong Adler-32
    s = R.random_samples(PX, 2, 16, seed=3)
    z = bytearray(zlib.compress(R.filtered(s, 2, 16, 0)))
    z[-1] ^= 0x40
    cases.append(("bad Adler-32", R.assemble(PX, PX, 2, 16, 0, bytes(z)), "Adler-32 mismatch"))
    return cases


def test_corrupt_streams_name_the_tile(matrix, ctx):
    good = [matrix[i] for i in (0, 37, 101)]
    for name, bad, msg in _corrupt_cases():
        files = [good[0][1], good[1][1], bad, good[2][1]]
        batch = PngBatch.from_bytes(files, convert_rgb=True)
        for b in (batch, batch.cuda()):
            out = np.zeros((4, PX, PX, 3), np.uint8)
            with pytest.raises(ValueError, match=rf"PNG tile 2: {msg}"):
                png.decode(b, ctx=ctx, out=out)
            for k, g in zip((0, 1, 3), good):
                np.testing.assert_array_equal(out[k], g[2], err_msg=name)


@pytest.fixture(scope="module")
def weights():
    from biscuit_b200.weights import random_init
    return random_init(seed=3)


@pytest.mark.parametrize("max_batch", [8, uq.BENCH_MICRO_BATCH])
def test_predict_with_the_option_equals_predict_uint8(matrix, weights, ctx, max_batch):
    rng = np.random.default_rng(max_batch)
    n = 37 if max_batch == 8 else 700
    pick = rng.integers(0, len(matrix), n)
    batch = PngBatch.from_bytes([matrix[i][1] for i in pick], convert_rgb=True)
    pixels = np.stack([matrix[i][2] for i in pick])
    iface = uq.UncertaintyInterface(weights, max_batch=max_batch, ctx=ctx)
    m_ref, s_ref = iface.predict(pixels, T=30, seed=5, tile_index_base=11)
    for b in (batch, batch.cuda()):
        m, s = iface(b, T=30, seed=5, tile_index_base=11)
        np.testing.assert_array_equal(m, m_ref)
        np.testing.assert_array_equal(s, s_ref)
    # without the option the same batch is rejected before the GPU runs
    with pytest.raises(ValueError, match=r"PNG tile \d+: (colour type|bit depth|interlaced)"):
        iface(PngBatch(batch.data, batch.offsets), T=30, seed=5)
    iface.close()


def test_predict_tfrecords_rgba_equals_predict_table(weights, ctx, tmp_path):
    import io

    from PIL import Image
    tiles = synth.tiles_u8(9, seed=13, n_slides=2)
    files = []
    for i, t in enumerate(tiles):                      # RGBA tiles as OpenSlide's read_region(...).save() writes them
        bio = io.BytesIO()
        Image.fromarray(np.dstack([t, np.full(t.shape[:2], 255 - 20 * i, np.uint8)]), "RGBA").save(bio, "PNG")
        files.append(bio.getvalue())
    slides = ["slide A"] * 5 + ["slide B"] * 4
    locs = [(10 * i, 3 * i) for i in range(9)]
    paths = [tmp_path / "a.tfrecords", tmp_path / "b.tfrecords"]
    jpeg_synth.write_tfrecord(paths[0], files[:5], slides[:5], locs[:5])
    jpeg_synth.write_tfrecord(paths[1], files[5:], slides[5:], locs[5:])
    iface = uq.UncertaintyInterface(weights, max_batch=8, ctx=ctx)
    labels = {"slide A": 0, "slide B": 1}
    df = uq.predict_tfrecords(iface, paths, y_true=labels, T=30, seed=2, png_convert_rgb=True)
    pixels = np.stack([R.decode(b) for b in files])
    np.testing.assert_array_equal(pixels, tiles)
    ref = uq.predict_table(iface, pixels, slides, y_true=[labels[s] for s in slides], T=30, seed=2)
    for col in ref.columns:
        np.testing.assert_array_equal(df[col].to_numpy(), ref[col].to_numpy(), err_msg=col)
    assert df["loc_x"].tolist() == [x for x, _ in locs]
    iface.close()
