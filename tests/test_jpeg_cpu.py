"""CPU tier of the compressed-tile input: TFRecord framing / CRC32C / Example parsing (bq_tfrecord_scan), the JPEG
marker parse that accepts or rejects a tile before anything runs on the GPU (bq_jpeg_inspect), and the numpy
restatement of libjpeg-turbo's decode (oracle/jpeg_ref.py) pinned to Pillow bit for bit."""
import itertools

import numpy as np
import pytest

from biscuit_b200 import jpeg, tfrecord
from biscuit_b200.jpeg import JpegBatch
from oracle import jpeg_ref, jpeg_synth, synth

QUALITIES = (50, 75, 90, 95, 100)
SAMPLINGS = ("4:4:4", "4:2:2", "4:2:0")
RESTARTS = ({}, {"restart_blocks": 1}, {"restart_blocks": 7}, {"restart_rows": 1})


# ------------------------------------------------------------------------------------------------------------------
# CRC32C and TFRecord framing
# ------------------------------------------------------------------------------------------------------------------
def test_crc32c_check_value():
    assert tfrecord.crc32c(b"123456789") == 0xE3069283
    assert jpeg_synth._crc32c(b"123456789") == 0xE3069283
    c = 0xE3069283
    assert tfrecord.masked_crc32c(b"123456789") == ((((c >> 15) | (c << 17)) & 0xFFFFFFFF) + 0xA282EAD8) & 0xFFFFFFFF
    rng = np.random.default_rng(0)
    for n in (0, 1, 7, 8, 9, 63, 1000):
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert tfrecord.crc32c(b) == jpeg_synth._crc32c(b)
        assert tfrecord.masked_crc32c(b) == jpeg_synth.masked_crc32c(b)


def _records(n=4, seed=0):
    rng = np.random.default_rng(seed)
    imgs = [rng.integers(0, 256, int(rng.integers(1, 3000)), dtype=np.uint8).tobytes() for _ in range(n)]
    slides = [f"slide-{i % 2}" for i in range(n)]
    locs = [(int(rng.integers(0, 10**6)), int(rng.integers(0, 10**6))) for _ in range(n)]
    return imgs, slides, locs


def test_tfrecord_round_trip(tmp_path):
    imgs, slides, locs = _records(5)
    p = tmp_path / "a.tfrecords"
    jpeg_synth.write_tfrecord(p, imgs, slides, locs)
    buf = p.read_bytes()
    image, slide, loc = tfrecord.scan(buf)
    assert len(image) == 5
    for i in range(5):
        assert buf[image[i, 0]:image[i, 1]] == imgs[i]
        assert buf[slide[i, 0]:slide[i, 1]].decode() == slides[i]
        assert tuple(loc[i]) == locs[i]
    batch, s, lx, ly = tfrecord.read([p, p])
    assert len(batch) == 10 and s == slides * 2
    assert [batch.tile(i) for i in range(10)] == imgs * 2
    assert list(lx) == [x for x, _ in locs] * 2 and list(ly) == [y for _, y in locs] * 2


def test_tfrecord_field_order_unknown_fields_and_non_ascii():
    img = b"\xff\xd8 not really a jpeg"
    name = "Schnitt-Ä_组织_🧫"
    feats = {"loc_y": 7, "slide": name.encode("utf-8"), "extra": 1.5, "image_raw": img, "loc_x": -3}
    recs = [jpeg_synth.tf_example(feats, order=o, packed=pk, extra_unknown=u)
            for o, pk, u in [(None, True, False), (["image_raw", "loc_x", "extra", "slide", "loc_y"], False, True)]]
    buf = b"".join(jpeg_synth.tfrecord_frame(r) for r in recs)
    image, slide, loc = tfrecord.scan(buf)
    for i in range(2):
        assert buf[image[i, 0]:image[i, 1]] == img
        assert buf[slide[i, 0]:slide[i, 1]].decode("utf-8") == name
        assert tuple(loc[i]) == (-3, 7)
    # keys are parameters; missing optional features are reported as absent
    image, slide, loc = tfrecord.scan(buf, image_key="slide", slide_key="nope", x_key="loc_y", y_key="absent")
    assert buf[image[0, 0]:image[0, 1]] == name.encode("utf-8")
    assert tuple(slide[0]) == (-1, -1) and loc[0, 0] == 7 and loc[0, 1] == tfrecord.LOC_MISSING
    with pytest.raises(ValueError, match="no bytes feature 'pixels'"):
        tfrecord.scan(buf, image_key="pixels")


def test_tfrecord_corruption_is_rejected():
    imgs, slides, locs = _records(3, seed=1)
    good = b"".join(jpeg_synth.tfrecord_frame(jpeg_synth.tf_example({"image_raw": i, "slide": s.encode()}))
                    for i, s in zip(imgs, slides))
    first_len = int.from_bytes(good[:8], "little")
    payload = bytearray(good)
    payload[12 + first_len // 2] ^= 0x01
    with pytest.raises(ValueError, match="record 0 .*payload CRC"):
        tfrecord.scan(bytes(payload))
    length = bytearray(good)
    length[0] ^= 0x04
    with pytest.raises(ValueError, match="length CRC"):
        tfrecord.scan(bytes(length))
    with pytest.raises(ValueError, match="record 2 .*truncated"):
        tfrecord.scan(good[:-5])
    import gzip
    import zlib
    with pytest.raises(ValueError, match="gzip"):
        tfrecord.scan(gzip.compress(good))
    with pytest.raises(ValueError, match="zlib"):
        tfrecord.scan(zlib.compress(good))


# ------------------------------------------------------------------------------------------------------------------
# JPEG marker parse
# ------------------------------------------------------------------------------------------------------------------
def test_inspect_accepts_every_encoding_of_the_matrix():
    tile = synth.tiles_u8(1, seed=4)[0]
    files = [jpeg_synth.jpeg_encode(tile, q, ss, opt, **rs)
             for q, ss, opt, rs in itertools.product(QUALITIES, SAMPLINGS, (False, True), RESTARTS)]
    assert len(files) == 120
    st = jpeg.inspect(JpegBatch.from_bytes(files))
    assert st.tolist() == [0] * 120


def _remove_segment(b, marker):
    i = 2
    while True:
        m, ln = b[i + 1], int.from_bytes(b[i + 2:i + 4], "big")
        if m == marker:
            return b[:i] + b[i + 2 + ln:]
        i += 2 + ln


def test_inspect_rejections_each_with_its_own_message():
    tile = synth.tiles_u8(1, seed=5)[0]
    good = jpeg_synth.jpeg_encode(tile, 90)
    sos = good.index(b"\xff\xda")
    cases = {
        "progressive": jpeg_synth.jpeg_encode(tile, 90, progressive=True),
        "grayscale": jpeg_synth.jpeg_encode(tile, 90, mode="L"),
        "CMYK": jpeg_synth.jpeg_encode(tile, 90, mode="CMYK"),
        "size": jpeg_synth.jpeg_encode(np.zeros((300, 300, 3), np.uint8), 90),
        "ends inside its headers": good[:sos - 40],
        "no DHT": _remove_segment(good, 0xC4),
    }
    batch = JpegBatch.from_bytes([good] + list(cases.values()))
    st = jpeg.inspect(batch)
    assert st[0] == 0
    msgs = [jpeg.status_message(s) for s in st[1:]]
    assert all(s != 0 for s in st[1:])
    assert len(set(msgs)) == len(msgs), msgs
    for (key, _), m in zip(cases.items(), msgs):
        assert key.lower() in m.lower(), (key, m)
    with pytest.raises(ValueError, match=r"JPEG tile 1: progressive"):
        jpeg.check(batch)


# ------------------------------------------------------------------------------------------------------------------
# the numpy restatement of the four decode stages, pinned to Pillow
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("subsampling", SAMPLINGS)
def test_jpeg_ref_matches_pil(subsampling):
    tiles = np.concatenate([synth.tiles_u8(1, seed=6), jpeg_synth.degenerate_tiles()[[1, 3, 4]]])
    for k, (q, opt, rs) in enumerate([(50, False, {}), (100, True, {"restart_blocks": 7}), (75, False, {"restart_rows": 1})]):
        for i, t in enumerate(tiles):
            b = jpeg_synth.jpeg_encode(t, q, subsampling, opt, **rs)
            np.testing.assert_array_equal(jpeg_ref.decode(b), jpeg_synth.pil_decode(b), err_msg=f"tile {i} q{q} {rs}")
