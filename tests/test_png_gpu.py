"""GPU tier of the PNG input: the CUDA PNG decoder equals Pillow byte for byte over the writer matrix (filters, zlib
levels, strategies, windows, flushes, IDAT sizes, ancillary chunks) and Pillow's own encodings, in one mixed batch;
every hand-made DEFLATE / Adler-32 / filter corruption raises ValueError naming the tile; `predict(PngBatch)` equals
`predict` on the decoded tiles bit for bit, and `predict_tfrecords` on PNG records equals `predict_table`."""
import numpy as np
import pytest

from biscuit_b200 import png, threshold, uq
from biscuit_b200.png import PngBatch
from oracle import jpeg_synth, png_synth, synth

pytestmark = pytest.mark.gpu

PX = synth.TILE_PX
ROW = 1 + 3 * PX


@pytest.fixture(scope="module")
def tiles():
    return np.concatenate([synth.tiles_u8(3, seed=21, n_slides=2), jpeg_synth.degenerate_tiles(),
                           png_synth.distance_tile()[None]])


@pytest.fixture(scope="module")
def matrix(tiles):
    """every encoding applied to every tile: (label, bytes, Pillow pixels, filter type per row or None)"""
    out = []
    for i, t in enumerate(tiles):
        for label, kw in png_synth.encodings():
            f = kw.get("filters", 0)
            filters = np.random.default_rng(kw.get("seed", 0)).integers(0, 5, PX) if isinstance(f, str) else [f] * PX
            b = png_synth.png_encode(t, **kw)
            out.append((f"{label} tile {i}", b, png_synth.pil_decode(b), filters))
        for k in png_synth.PIL_LEVELS:
            b = png_synth.pil_encode(t, k)
            out.append((f"Pillow level {k} tile {i}", b, png_synth.pil_decode(b), None))
    return out


def _first_mismatch(got, want, labels, filters):
    bad = np.flatnonzero((got != want).reshape(len(got), -1).any(1))
    if not bad.size:
        return None
    lines = [f"{bad.size} of {len(got)} tiles differ"]
    for t in bad[:5]:
        yx = np.argwhere(got[t] != want[t])
        y, x, c = yx[0]
        ft = "?" if filters[t] is None else int(filters[t][y])
        lines.append(f"  {labels[t]}: {len(yx)} values differ; first at row {y} column {x} channel {c} (filter type "
                     f"{ft}): got {got[t][y, x]} want {want[t][y, x]}")
    return "\n".join(lines)


def test_decode_matrix_bit_exact(matrix, ctx):
    labels, files, want, filters = zip(*matrix)
    got = png.decode(PngBatch.from_bytes(files), ctx=ctx)          # every encoding mixed in one batch
    msg = _first_mismatch(got, np.stack(want), labels, filters)
    assert msg is None, msg


@pytest.mark.parametrize("n", [1, 3, 503, 1200])
def test_decode_batch_sizes_host_and_device(matrix, ctx, n):
    import torch
    rng = np.random.default_rng(n)
    pick = rng.integers(0, len(matrix), n)
    want = np.stack([matrix[i][2] for i in pick])
    batch = PngBatch.from_bytes([matrix[i][1] for i in pick])
    for b in (batch, batch.cuda()):
        np.testing.assert_array_equal(png.decode(b, ctx=ctx), want)
        out = torch.empty((n, PX, PX, 3), dtype=torch.uint8, device="cuda")
        png.decode(b, ctx=ctx, out=out)
        np.testing.assert_array_equal(out.cpu().numpy(), want)


def test_crafted_streams_rejected_with_tile_index(tiles, ctx):
    raw = png_synth.filter_rows(tiles[0], np.arange(PX) % 5)
    good = [png_synth.pil_encode(t) for t in tiles[:3]]
    for name, (z, status, _) in png_synth.crafted_streams(raw, ROW).items():
        f = png_synth.assemble(PX, PX, z, idat_size=8192)
        batch = PngBatch.from_bytes([good[0], f, good[2]])
        if status is None:
            np.testing.assert_array_equal(png.decode(batch, ctx=ctx)[1], png_synth.pil_decode(f), err_msg=name)
            continue
        for b in (batch, batch.cuda()):
            with pytest.raises(ValueError, match=rf"PNG tile 1: {status}"):
                png.decode(b, ctx=ctx)
    # an IDAT run that ends inside the file's last chunk
    cut = good[1][:len(good[1]) - 40]
    with pytest.raises(ValueError, match=r"PNG tile 2: truncated data"):
        png.decode(PngBatch.from_bytes([good[0], good[2], cut]), ctx=ctx)
    np.testing.assert_array_equal(png.decode(PngBatch.from_bytes(good), ctx=ctx), tiles[:3])


def test_header_rejection_before_launch(tiles, ctx):
    good = png_synth.pil_encode(tiles[0])
    gray = png_synth.pil_encode(tiles[0], mode="L")
    launches = ctx.launches
    with pytest.raises(ValueError, match=r"PNG tile 1: colour type"):
        png.decode(PngBatch.from_bytes([good, gray]), ctx=ctx)
    assert ctx.launches == launches


@pytest.fixture(scope="module")
def weights():
    from biscuit_b200.weights import random_init
    return random_init(seed=3)


@pytest.mark.parametrize("max_batch", [8, uq.BENCH_MICRO_BATCH])
@pytest.mark.parametrize("normalizer", [None, "reinhard_fast"])
def test_predict_png_equals_predict_uint8(matrix, weights, ctx, max_batch, normalizer):
    rng = np.random.default_rng(max_batch)
    n = 37 if max_batch == 8 else 700
    pick = rng.integers(0, len(matrix), n)
    batch = PngBatch.from_bytes([matrix[i][1] for i in pick])
    pixels = np.stack([matrix[i][2] for i in pick])
    iface = uq.UncertaintyInterface(weights, max_batch=max_batch, ctx=ctx, normalizer=normalizer)
    m_ref, s_ref = iface.predict(pixels, T=30, seed=5, tile_index_base=11)
    for b in (batch, batch.cuda()):
        m, s = iface(b, T=30, seed=5, tile_index_base=11)
        np.testing.assert_array_equal(m, m_ref)
        np.testing.assert_array_equal(s, s_ref)
    iface.close()


def test_predict_tfrecords_png_equals_predict_table(tiles, weights, ctx, tmp_path):
    paths, all_files, all_slides, all_locs = [], [], [], []
    k = 0
    for f, (slide, count) in enumerate([("slide A", 5), ("slide B", 4), ("slide A", 6)]):
        files = [png_synth.pil_encode(tiles[(k + j) % len(tiles)], (1, 6, 9)[f]) for j in range(count)]
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
    df = uq.predict_tfrecords(iface, paths, y_true=labels, T=30, seed=2)
    pixels = np.stack([png_synth.pil_decode(b) for b in all_files])
    ref = uq.predict_table(iface, pixels, all_slides, y_true=[labels[s] for s in all_slides], T=30, seed=2)
    for col in ref.columns:
        np.testing.assert_array_equal(df[col].to_numpy(), ref[col].to_numpy(), err_msg=col)
    assert df["loc_x"].tolist() == [x for x, _ in all_locs] and df["loc_y"].tolist() == [y for _, y in all_locs]
    threshold.apply(df.drop(columns=["loc_x", "loc_y"]), 0.5, 0.5)
    iface.close()
