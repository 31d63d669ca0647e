"""GPU tier: the route of float32 tiles the caller already standardised (`predict` on float32 ->
bq_predict_uq_standardized, the reference's literal call), which runs its own first layer (conv1_kernel<float>, CUDA
cores, no tile statistics) and its own double-buffered float staging.

  * block1_conv1 on that route against the float64 bound of conv1_f32_ref, on standardised, raw, TF-style and +-1e4
    inputs, and block1_conv2 on its output within its own bound; a partial micro-batch gives the same bits;
  * host (pageable, pinned) and device tiles, a device view at a one-tile offset, two micro-batch sizes, tile-by-tile
    calls and a staging buffer that grows between calls all give bit-identical results;
  * float and uint8 calls on one interface do not disturb each other, and a stain normaliser does not touch float input;
  * a NaN or +-Inf fails the call with ValueError naming the tile, and leaves the interface as it was;
  * uint8 tiles read in place from device memory at every base alignment equal the host-staged call.
"""
import numpy as np
import pytest
import torch

from helpers import float_tile_sets, tf_standardize
from oracle import synth, xception_ops as XO, xception_uq as X

pytestmark = pytest.mark.gpu

T = 10
SEED = 77
TILE = 299 * 299 * 3


@pytest.fixture(scope="module")
def weights():
    return X.make_weights(seed=1)


@pytest.fixture(scope="module")
def opw(weights):
    return XO.OpWeights(weights, device="cuda")


@pytest.fixture(scope="module")
def sets(weights):
    return float_tile_sets(weights)


@pytest.fixture(scope="module")
def pool(sets):
    """19 = 2 * 8 + 3 float tiles: synthetic and degenerate tiles standardised by the oracle, TF-style ones"""
    extra = tf_standardize(synth.tiles_u8(3, seed=5, n_slides=1))
    return np.ascontiguousarray(np.concatenate([sets["oracle"], sets["tf"], extra]))


def _iface(weights, max_batch, **kw):
    from biscuit_b200.uq import UncertaintyInterface
    return UncertaintyInterface(weights, max_batch=max_batch, **kw)


@pytest.fixture(scope="module")
def it8(weights):
    it = _iface(weights, 8)
    yield it
    it.close()


@pytest.fixture(scope="module")
def it4(weights):
    it = _iface(weights, 4)
    yield it
    it.close()


def _same(a, b, what):
    for x, y, name in zip(a, b, ("mean", "std", "features")):
        bad = np.nonzero((x != y).reshape(len(x), -1).any(1))[0]
        assert x.tobytes() == y.tobytes(), f"{what}: {name} of tiles {bad} differ"


# ------------------------------------------------------------------------------------------------------------------
# block1_conv1 / block1_conv2 within their bounds
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["oracle", "tf", "raw", "big"])
def test_float_route_first_layers_within_bound(it8, sets, opw, name):
    tiles = sets[name]
    conv1, conv2 = XO.plan()[:2]
    y1 = it8.debug_stage(tiles, "block1_conv1")
    rep = XO.check(f"block1_conv1[{name}]", torch.from_numpy(y1).cuda(), XO.op_ref(conv1, {"tiles": tiles}, opw), relu=True)
    print(f"float route block1_conv1 [{name}]: single-valued {rep['single']:.4f}, "
          f"max |y - z| / (E + half ulp) {rep['ratio']:.3f}")
    assert rep["n_fail"] == 0, XO.describe(rep)
    assert rep["single"] >= XO.SINGLE_FLOOR["block1_conv1_f32"], rep["single"]
    if name == "oracle":                     # constant tiles standardise to exact zeros: every output is bf16(ReLU(shift))
        want = XO.rn_bf16(torch.clamp_min(opw.affine["block1_conv1"][1], 0.0)).cpu().numpy()
        assert (y1[4:6] == want).all()
    y2 = it8.debug_stage(tiles, "block1_conv2")
    rep2 = XO.check(f"block1_conv2[{name}]", torch.from_numpy(y2).cuda(),
                    XO.op_ref(conv2, {"block1_conv1": torch.from_numpy(y1).cuda()}, opw), relu=True)
    print(f"float route block1_conv2 [{name}]: single-valued {rep2['single']:.4f}, max ratio {rep2['ratio']:.3f}")
    assert rep2["n_fail"] == 0, XO.describe(rep2)
    # a partial micro-batch gives the same bits as the same tiles in the full one
    for tag, y in (("block1_conv1", y1), ("block1_conv2", y2)):
        y3 = it8.debug_stage(tiles[:3], tag)
        assert y3.tobytes() == y[:3].tobytes(), f"{tag}: 3- and 8-tile micro-batches differ"


def test_debug_stage_dispatches_on_dtype(it8, sets):
    """float32 from numpy, a CPU or a CUDA tensor takes the float route (not a cast to bytes); uint8 the raw route;
    anything else is refused"""
    t = sets["raw"][:2]
    ref = it8.debug_stage(t, "block1_conv1")
    assert ref.tobytes() == it8.debug_stage(torch.from_numpy(t), "block1_conv1").tobytes()
    assert ref.tobytes() == it8.debug_stage(torch.from_numpy(t).cuda(), "block1_conv1").tobytes()
    u8 = it8.debug_stage(t.astype(np.uint8), "block1_conv1")
    assert u8.tobytes() != ref.tobytes()                     # raw 0-255 floats are not standardised; uint8 tiles are
    for bad in (t.astype(np.float64), t.astype(np.int32), torch.from_numpy(t).half()):
        with pytest.raises(TypeError):
            it8.debug_stage(bad, "block1_conv1")
    with pytest.raises(ValueError):
        it8.debug_stage(t[:, :298], "block1_conv1")


# ------------------------------------------------------------------------------------------------------------------
# staging and memory kinds
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [4, 8])
def test_float_route_staging_and_memory_kinds(weights, pool, B):
    """2 B + 3 tiles (two full micro-batches and a partial one) from every kind of memory, on a fresh interface whose
    staging buffer is sized by a 1-tile call and grows on the next; then each tile alone at its global index"""
    n = 2 * B + 3
    tiles = np.ascontiguousarray(pool[:n])
    it = _iface(weights, B)
    try:
        first = it.predict(tiles[:1], T=T, seed=SEED, return_features=True)        # staging sized for one tile
        ref = it.predict(tiles, T=T, seed=SEED, return_features=True)               # grows to B tiles
        _same(first, [a[:1] for a in ref], "1-tile call vs the first tile of the batch")
        again = it.predict(tiles[:1], T=T, seed=SEED, return_features=True)
        _same(again, first, "1-tile call after the batch")
        dev = torch.from_numpy(tiles).cuda()
        buf = torch.zeros((n + 1, 299, 299, 3), dtype=torch.float32, device="cuda")
        buf[1:] = dev
        view = buf[1:]                                                             # storage offset of one tile
        assert view.is_contiguous() and view.data_ptr() - buf.data_ptr() == TILE * 4
        for what, t in (("pinned", torch.from_numpy(tiles).pin_memory()), ("cuda", dev), ("cuda view", view)):
            _same(it.predict(t, T=T, seed=SEED, return_features=True), ref, what)
        for i in range(n):
            one = it.predict(tiles[i:i + 1], T=T, seed=SEED, tile_index_base=i, return_features=True)
            _same(one, [a[i:i + 1] for a in ref], f"tile {i} alone")
    finally:
        it.close()
    # the same tiles at the other micro-batch size: the first 11 tiles are common to both parametrisations
    other = _iface(weights, 12 - B)
    try:
        _same(other.predict(tiles[:11], T=T, seed=SEED, return_features=True), [a[:11] for a in ref],
              f"max_batch {12 - B} vs {B}")
    finally:
        other.close()


# ------------------------------------------------------------------------------------------------------------------
# interleaving with the uint8 route, and the normaliser
# ------------------------------------------------------------------------------------------------------------------
def test_float_and_uint8_calls_do_not_disturb_each_other(weights, it4, pool):
    """the float flag is reset after a float call and the captured graph of the full micro-batches serves both routes:
    a uint8 call between two float calls (and the reverse) changes nothing; an interface with the Reinhard
    normaliser gives the float route's results bit for bit, since float tiles skip the normaliser"""
    f = pool[:11]
    u = np.concatenate([synth.tiles_u8(8, seed=3, n_slides=2), synth.tiles_u8(3, seed=4)])
    f1 = it4.predict(f, T=T, seed=SEED, return_features=True)
    u1 = it4.predict(u, T=T, seed=SEED, return_features=True)
    f2 = it4.predict(f, T=T, seed=SEED, return_features=True)
    u2 = it4.predict(u, T=T, seed=SEED, return_features=True)
    _same(f2, f1, "float call after a uint8 call")
    _same(u2, u1, "uint8 call after a float call")
    it = _iface(weights, 4, normalizer="reinhard_fast")
    try:
        _same(it.predict(f, T=T, seed=SEED, return_features=True), f1, "float route with the normaliser set")
        assert it.predict(u[:4], T=T, seed=SEED)[0].tobytes() != u1[0][:4].tobytes()     # the normaliser is on
    finally:
        it.close()


# ------------------------------------------------------------------------------------------------------------------
# non-finite input
# ------------------------------------------------------------------------------------------------------------------
def test_non_finite_float_input_is_an_error(it4, pool):
    """NaN, +Inf, -Inf at the first, the last and an interior value of tile k = 5 (second micro-batch at max_batch 4),
    from host and device memory: ValueError naming tile 5, the other tiles' results still written; two bad tiles name
    the smaller index; afterwards the interface reproduces its results bit for bit"""
    tiles = np.ascontiguousarray(pool[:11])
    k = 5
    ref = it4.predict(tiles, T=T, seed=SEED)
    nc = ref[0].shape[1]
    ok = np.arange(len(tiles)) != k
    for val in (np.nan, np.inf, -np.inf):
        for pos in (0, TILE - 1, 150 * 299 * 3 + 150 * 3 + 1):
            bad = tiles.copy()
            bad[k].reshape(-1)[pos] = val
            for where, t in (("host", bad), ("cuda", torch.from_numpy(bad).cuda())):
                m = np.full((len(tiles), nc), -1, np.float32)
                s = np.full((len(tiles), nc), -1, np.float32)
                with pytest.raises(ValueError, match=f"tile {k}: non-finite value"):
                    it4.predict(t, T=T, seed=SEED, out_mean=m, out_std=s)
                assert m[ok].tobytes() == ref[0][ok].tobytes() and s[ok].tobytes() == ref[1][ok].tobytes(), (val, pos, where)
    bad = tiles.copy()
    bad[9, 7, 7, 2] = np.nan
    bad[k, 0, 0, 0] = np.inf
    with pytest.raises(ValueError, match=f"tile {k}: non-finite value"):
        it4.predict(bad, T=T, seed=SEED)
    after = it4.predict(tiles, T=T, seed=SEED)
    _same(after, ref, "after the failed calls")


# ------------------------------------------------------------------------------------------------------------------
# uint8 tiles in device memory at every base alignment
# ------------------------------------------------------------------------------------------------------------------
def test_device_uint8_tiles_at_every_alignment(it4):
    """tile_stats_kernel splits each tile into an unaligned head, 16-byte vectors and a tail, and conv1_tc_kernel copies
    an aligned superset of its patch: a byte view at offsets 0-15 into a buffer with 64 bytes of noise on either side
    must give the host-staged results bit for bit"""
    tiles = np.ascontiguousarray(synth.tiles_u8(6, seed=8, n_slides=2))
    ref = it4.predict(tiles, T=T, seed=SEED, return_features=True)
    flat = torch.from_numpy(tiles.reshape(-1)).cuda()
    g = torch.Generator(device="cuda").manual_seed(3)
    for off in range(16):
        buf = torch.randint(0, 256, (64 + off + flat.numel() + 64,), dtype=torch.uint8, device="cuda", generator=g)
        buf[64 + off:64 + off + flat.numel()] = flat
        view = buf[64 + off:64 + off + flat.numel()].view(6, 299, 299, 3)
        _same(it4.predict(view, T=T, seed=SEED, return_features=True), ref, f"device tiles at offset {off}")
