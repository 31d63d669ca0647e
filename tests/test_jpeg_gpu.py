"""GPU tier of the compressed-tile input: the CUDA JPEG decoder equals Pillow (libjpeg-turbo's default decode) byte for
byte over the quality x sampling x table x restart matrix, `predict(JpegBatch)` equals `predict` on the Pillow-decoded
tiles bit for bit, `predict_tfrecords` equals `predict_table`, and corrupt entropy-coded data raises ValueError."""
import itertools

import numpy as np
import pytest

from biscuit_b200 import jpeg, threshold, uq
from biscuit_b200.jpeg import JpegBatch
from oracle import jpeg_synth, synth

pytestmark = pytest.mark.gpu

QUALITIES = (50, 75, 90, 95, 100)
SAMPLINGS = ("4:4:4", "4:2:2", "4:2:0")
RESTARTS = ({}, {"restart_blocks": 1}, {"restart_blocks": 7}, {"restart_rows": 1})
MCU = {"4:4:4": (8, 8), "4:2:2": (8, 16), "4:2:0": (16, 16)}


@pytest.fixture(scope="module")
def tiles():
    return np.concatenate([synth.tiles_u8(3, seed=21, n_slides=2), jpeg_synth.degenerate_tiles()])


@pytest.fixture(scope="module")
def matrix(tiles):
    """every encoding of the matrix applied to every tile: (label, sampling, bytes, Pillow pixels)"""
    out = []
    for q, ss, opt, rs in itertools.product(QUALITIES, SAMPLINGS, (False, True), RESTARTS):
        for i, t in enumerate(tiles):
            b = jpeg_synth.jpeg_encode(t, q, ss, opt, **rs)
            out.append((f"q{q} {ss} optimize={opt} {rs} tile {i}", ss, b, jpeg_synth.pil_decode(b)))
    return out


def _first_mismatch(got, want, labels, samplings):
    bad = np.flatnonzero((got != want).reshape(len(got), -1).any(1))
    if not bad.size:
        return None
    lines = [f"{bad.size} of {len(got)} tiles differ"]
    for t in bad[:5]:
        yx = np.argwhere(got[t] != want[t])
        mh, mw = MCU[samplings[t]]
        y, x, c = yx[0]
        lines.append(f"  {labels[t]}: {len(yx)} values differ; first at pixel ({y}, {x}) component {c} MCU "
                     f"({y // mh}, {x // mw}): got {got[t][y, x]} want {want[t][y, x]}")
    return "\n".join(lines)


def test_decode_matrix_bit_exact(matrix, ctx):
    labels, samplings, files, want = zip(*matrix)
    got = jpeg.decode(JpegBatch.from_bytes(files), ctx=ctx)         # every encoding mixed in one batch
    msg = _first_mismatch(got, np.stack(want), labels, samplings)
    assert msg is None, msg
    st = jpeg.last_stats(ctx)
    assert st["tiles"] == len(files) and st["subsequences"] >= len(files)


@pytest.mark.parametrize("n", [1, 3, 503, 1200])
def test_decode_batch_sizes_host_and_device(matrix, ctx, n):
    import torch
    rng = np.random.default_rng(n)
    pick = rng.integers(0, len(matrix), n)
    files = [matrix[i][2] for i in pick]
    want = np.stack([matrix[i][3] for i in pick])
    batch = JpegBatch.from_bytes(files)
    np.testing.assert_array_equal(jpeg.decode(batch, ctx=ctx), want)
    out = torch.empty((n, 299, 299, 3), dtype=torch.uint8, device="cuda")
    jpeg.decode(batch.cuda(), ctx=ctx, out=out)
    np.testing.assert_array_equal(out.cpu().numpy(), want)


def _entropy_start(b):
    sos = b.index(b"\xff\xda")
    return sos + 2 + int.from_bytes(b[sos + 2:sos + 4], "big")


def test_corrupt_entropy_data_raises_with_tile_index(tiles, ctx):
    good = [jpeg_synth.jpeg_encode(t, 90) for t in tiles[:3]]
    s = _entropy_start(good[1])
    cut = s + (len(good[1]) - s) // 2
    while good[1][cut - 1] == 0xFF:                       # cut between two coded bytes, not inside FF00 stuffing
        cut -= 1
    truncated = good[1][:cut] + b"\xff\xd9"
    # a run of 1-bits longer than any code: no table holds it
    at = _entropy_start(good[2]) + 40
    while good[2][at - 1] == 0xFF:
        at += 1
    invalid = good[2][:at] + b"\xff\x00" * 4 + good[2][at:]
    with pytest.raises(ValueError, match=r"JPEG tile 1: entropy-coded data truncated"):
        jpeg.decode(JpegBatch.from_bytes([good[0], truncated, good[2]]), ctx=ctx)
    with pytest.raises(ValueError, match=r"JPEG tile 2: invalid Huffman code"):
        jpeg.decode(JpegBatch.from_bytes([good[0], good[1], invalid]), ctx=ctx)
    np.testing.assert_array_equal(jpeg.decode(JpegBatch.from_bytes(good), ctx=ctx),
                                  np.stack([jpeg_synth.pil_decode(b) for b in good]))


def test_header_rejection_before_launch(tiles, ctx):
    good = jpeg_synth.jpeg_encode(tiles[0], 90)
    prog = jpeg_synth.jpeg_encode(tiles[0], 90, progressive=True)
    launches = ctx.launches
    with pytest.raises(ValueError, match=r"JPEG tile 1: progressive"):
        jpeg.decode(JpegBatch.from_bytes([good, prog]), ctx=ctx)
    assert ctx.launches == launches


@pytest.fixture(scope="module")
def weights():
    from biscuit_b200.weights import random_init
    return random_init(seed=3)


@pytest.mark.parametrize("max_batch", [8, uq.BENCH_MICRO_BATCH])
@pytest.mark.parametrize("normalizer", [None, "reinhard_fast"])
def test_predict_jpeg_equals_predict_uint8(matrix, weights, ctx, max_batch, normalizer):
    rng = np.random.default_rng(max_batch)
    n = 37 if max_batch == 8 else 700
    pick = rng.integers(0, len(matrix), n)
    batch = JpegBatch.from_bytes([matrix[i][2] for i in pick])
    pixels = np.stack([matrix[i][3] for i in pick])
    iface = uq.UncertaintyInterface(weights, max_batch=max_batch, ctx=ctx, normalizer=normalizer)
    m_ref, s_ref = iface.predict(pixels, T=30, seed=5, tile_index_base=11)
    for b in (batch, batch.cuda()):
        m, s = iface.predict(b, T=30, seed=5, tile_index_base=11)
        np.testing.assert_array_equal(m, m_ref)
        np.testing.assert_array_equal(s, s_ref)
    iface.close()


def test_predict_tfrecords_equals_predict_table(tiles, weights, ctx, tmp_path):
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
    df = uq.predict_tfrecords(iface, paths, y_true=labels, T=30, seed=2)
    pixels = np.stack([jpeg_synth.pil_decode(b) for b in all_files])
    ref = uq.predict_table(iface, pixels, all_slides, y_true=[labels[s] for s in all_slides], T=30, seed=2)
    for col in ref.columns:
        np.testing.assert_array_equal(df[col].to_numpy(), ref[col].to_numpy(), err_msg=col)
    assert df["loc_x"].tolist() == [x for x, _ in all_locs] and df["loc_y"].tolist() == [y for _, y in all_locs]
    threshold.apply(df.drop(columns=["loc_x", "loc_y"]), 0.5, 0.5)
    iface.close()
