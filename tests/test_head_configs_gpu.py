"""GPU tier: the fused MC-dropout head (head_sm100.cuh) and hidden_0 on every configuration the library accepts, each
checked against the float64 reference with a proven error bound (oracle/xception_ops.py: head_ref, hidden0_ref) from
the GPU's own hidden_0 output and injected masks, and the kernels' own Philox stream bit-identical to those masks.

Cases: hidden widths 64 .. 1024 (one box of W2 rows below 256, a partly out-of-range second 256-column MMA block at
320 and 576, two 512-column halves above 512) with 2 .. 8 classes; all seven dropout placements; rates 0, 0.1, 0.5 and
0.9; T from 1 to 4096 (up to 128 sample chunks merged) with T changing on one interface; CTAs that run two four-tile
groups (1006 tiles in one head launch); and the seams between head batches.
"""
import numpy as np
import pytest
import torch

from helpers import degenerate_tiles
from oracle import synth, xception_ops as XO, xception_uq as X

pytestmark = pytest.mark.gpu

SEED = 77
DEFAULT = (False, True, True)
ALL_SITES = [tuple(bool(m >> i & 1) for i in range(3)) for m in range(1, 8)]


@pytest.fixture(scope="module")
def tiles():
    """4 synthetic tiles + 4 degenerate ones = max_batch"""
    return np.ascontiguousarray(np.concatenate([synth.tiles_u8(4, seed=0, n_slides=3), degenerate_tiles()]))


@pytest.fixture(scope="module")
def features():
    """pooled features of every configuration: the backbone weights of random_init do not depend on W or C"""
    return {}


def make_iface(W=1024, C=2, sites=DEFAULT, rate=0.1, max_batch=8):
    from biscuit_b200.hp import nature2022
    from biscuit_b200.uq import UncertaintyInterface
    from biscuit_b200.weights import random_init
    w = random_init(seed=1, hidden_width=W, n_classes=C)
    cfg = nature2022.replace(hidden_layer_width=W, n_classes=C, dropout_sites=sites, dropout=rate)
    return UncertaintyInterface(w, config=cfg, max_batch=max_batch), XO.HeadWeights(w, device="cuda")


def masks_for(n, T, W, rate, sites, tile_index_base=0):
    enabled = [i for i, on in enumerate(sites) if on]
    return X.keep_masks(n, T, 2048 if sites[0] else W, rate, SEED, tile_index_base=tile_index_base, sites=enabled)


def check_case(it, hw, tiles, T, tag, features=None):
    """predict with injected masks; hidden_0 and the head within the bound; the Philox stream gives the same bits"""
    cfg = it.config
    W, rate, sites = cfg.hidden_layer_width, cfg.dropout, cfg.dropout_sites
    n = len(tiles)
    masks = masks_for(n, T, W, rate, sites)
    mean, std, feats = it.predict(tiles, T=T, masks=masks, return_features=True)
    if features is not None:
        ref = features.setdefault("ref", feats)
        assert ref.tobytes() == feats.tobytes(), f"{tag}: features differ from the first configuration's"
    h1 = torch.from_numpy(it.debug_h1(n)).cuda()
    k0 = masks[:, :, 0] if sites[0] else None
    z, E = XO.hidden0_ref(torch.from_numpy(feats).cuda(), hw, k0=k0, rate=rate)
    rep = XO.check("hidden_0", h1.reshape(-1, W), ("bound", (z.reshape(-1, W), E.reshape(-1, W))), relu=True)
    assert rep["n_fail"] == 0, f"{tag}: " + XO.describe(rep)
    assert rep["single"] >= XO.SINGLE_FLOOR["hidden_0"], (tag, rep["single"])
    h = XO.head_ref(h1, masks, hw, rate, sites)
    hr = XO.head_report(mean, std, h)
    print(f"{tag}: hidden_0 single-valued {rep['single']:.3f} max |y-z|/E {rep['ratio']:.3f}; head mean width "
          f"{hr['width']:.2e}, |d mean|/half-width {hr['ratio_mean']:.3f}, |d std|/allowed {hr['ratio_std']:.3f}")
    assert hr["n_fail_mean"] == 0 and hr["n_fail_std"] == 0, XO.describe_head(tag, hr)
    # sharp enough that a mask on the neighbouring unit (a 5e-3 .. 2e-2 move of the mean) fails; a class's interval
    # collects the uncertainty of its C - 1 logit differences, so 8 classes widen it (up to ~2.3e-3 on these tiles)
    if rate <= 0.5:
        assert hr["width"] <= (2e-3 if cfg.n_classes <= 3 else 3e-3), (tag, hr["width"])
    own = it.predict(tiles, T=T, seed=SEED)
    assert own[0].tobytes() == mean.tobytes() and own[1].tobytes() == std.tobytes(), \
        f"{tag}: the Philox stream differs from the injected masks"
    return mean, std


GEOMETRY = [(64, 8), (128, 2), (192, 3), (256, 2), (320, 5), (576, 8), (1024, 3), (1024, 8)]


@pytest.mark.parametrize("W,C", GEOMETRY, ids=[f"W{w}-C{c}" for w, c in GEOMETRY])
def test_geometry(tiles, features, W, C):
    """hidden widths below one 256-row box, with a partial second MMA block, one or two halves; 2 .. 8 classes"""
    it, hw = make_iface(W, C)
    try:
        check_case(it, hw, tiles, 33, f"W={W} C={C} T=33", features)
    finally:
        it.close()


@pytest.mark.parametrize("sites", ALL_SITES, ids=["s" + "".join("1" if x else "0" for x in s) for s in ALL_SITES])
def test_placement(tiles, features, sites):
    """every non-empty dropout placement at rate 0.1; site 0 makes hidden_0 per sample"""
    it, hw = make_iface(sites=sites)
    try:
        check_case(it, hw, tiles, 33, f"sites={sites} T=33", features)
    finally:
        it.close()


@pytest.mark.parametrize("rate", [0.0, 0.5, 0.9])
def test_rate(tiles, features, rate):
    """rates at both ends; at rate 0 every sample is the same, so the std is within the slack of 0, and exactly 0 where
    the chunk sums are exact (T a power of two <= 32, or T = 1: a lone sample in its chunk)"""
    it, hw = make_iface(rate=rate)
    try:
        for T in ((1, 16, 32, 33) if rate == 0.0 else (33,)):
            mean, std = check_case(it, hw, tiles, T, f"rate={rate} T={T}", features)
            if rate == 0.0:
                assert np.abs(std).max() <= 1e-6, (T, np.abs(std).max())
                if T <= 32 and T & (T - 1) == 0:
                    assert not std.any(), (T, std)
    finally:
        it.close()


@pytest.fixture(scope="module")
def t_iface():
    it, hw = make_iface()
    yield it, hw
    it.close()


# 7 -> 4096 -> 33 -> 4096 on one interface: the head buffers grow (head_T_cap) and the descriptors are rebuilt
T_SEQUENCE = [7, 4096, 33, 4096, 1, 2, 31, 32, 64, 100, 1000]


@pytest.mark.parametrize("i", range(len(T_SEQUENCE)), ids=[f"{i}-T{t}" for i, t in enumerate(T_SEQUENCE)])
def test_sample_count(tiles, t_iface, i):
    """T from 1 to 4096 with the default placement: 1 .. 128 sample chunks merged with Chan's formula"""
    it, hw = t_iface
    check_case(it, hw, tiles, T_SEQUENCE[i], f"T={T_SEQUENCE[i]} (call {i})")


def test_multi_group_ctas(tiles):
    """max_batch = the bench micro-batch: 1006 tiles make one head batch and one head launch of 252 four-tile groups on
    148 SMs, so most CTAs run a second group; every tile within the bound"""
    from biscuit_b200.uq import BENCH_MICRO_BATCH
    n, T = 2 * BENCH_MICRO_BATCH, 100
    it, hw = make_iface(max_batch=BENCH_MICRO_BATCH)
    try:
        big = np.ascontiguousarray(np.resize(tiles, (n,) + tiles.shape[1:]))
        check_case(it, hw, big, T, f"n={n} T={T}")
    finally:
        it.close()


def test_head_batch_seams(tiles):
    """max_batch = 8: 1200 tiles run as head batches of 592, 592 and 16 tiles.  With injected masks from host memory and
    from device memory, every tile's mean and std equal, bit for bit, the same tile run alone with its own mask slice
    and tile_index_base"""
    n, T = 1200, 7
    it, _ = make_iface()
    try:
        big = np.ascontiguousarray(np.resize(tiles, (n,) + tiles.shape[1:]))
        masks = masks_for(n, T, 1024, 0.1, DEFAULT)
        mean, std = it.predict(big, T=T, masks=masks)
        mean_d, std_d = it.predict(big, T=T, masks=torch.from_numpy(masks).cuda())
        assert mean_d.tobytes() == mean.tobytes() and std_d.tobytes() == std.tobytes(), "device masks differ from host"
        bad = []
        for i in range(n):
            m1, s1 = it.predict(big[i:i + 1], T=T, masks=masks[i:i + 1], tile_index_base=i)
            if m1.tobytes() != mean[i:i + 1].tobytes() or s1.tobytes() != std[i:i + 1].tobytes():
                bad.append(i)
        assert not bad, f"{len(bad)} tiles differ from their lone run; first {bad[:8]} (head batch {[b // 592 for b in bad[:8]]})"
    finally:
        it.close()


def test_rejected_configurations():
    """widths beyond the fused head's 1024 fail at creation, not at the first predict"""
    from biscuit_b200.errors import NativeLibraryError
    with pytest.raises(NativeLibraryError, match="width <= 1024"):
        make_iface(W=1088)
