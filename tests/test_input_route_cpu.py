"""CPU tier: the float64 reference and error bound of block1_conv1 on float32 tiles the caller already standardised
(oracle/xception_ops.py: conv1_f32_ref, the arithmetic of conv1_kernel<float> in layers.cuh), checked without a GPU.

  * not too tight: an fp32 emulation of the kernel (27 fmas from 0 in (ky, kx, ci) order, RN(* scale), RN(+ shift), ReLU,
    bf16) passes on every input set of tests/test_input_route_gpu.py, and so do variants that sum in reverse order or
    round the product before the add;
  * not too loose: kernel-like bugs fail, and the failure histogram points at the rows or channels they touch.
"""
import numpy as np
import pytest
import torch

from helpers import float_tile_sets
from oracle import xception_ops as XO, xception_uq as X

TAPS = [(ky, kx, ci) for ky in range(3) for kx in range(3) for ci in range(3)]
CONV1 = XO.plan()[0]


@pytest.fixture(scope="module")
def weights():
    return X.make_weights(seed=1)


@pytest.fixture(scope="module")
def ow(weights):
    return XO.OpWeights(weights)


@pytest.fixture(scope="module")
def sets(weights):
    return float_tile_sets(weights)


@pytest.fixture(scope="module")
def refs(sets, ow):
    return {k: XO.op_ref(CONV1, {"tiles": t}, ow) for k, t in sets.items()}


def emulate(tiles, ow, order=TAPS, fused=True, w=None, relu=lambda y: torch.clamp_min(y, 0.0)):
    """conv1_kernel<float> in fp32: acc = RN(x * w + acc) over the 27 taps in `order` (the product is exact in float64, so
    RN32(float64 sum) is the fma up to a rare double rounding), or RN(acc + RN(x * w)) with fused=False; then
    RN(acc * scale), RN(+ shift), `relu`, bf16"""
    x = torch.from_numpy(np.ascontiguousarray(tiles)).to(torch.float64)
    w = (ow.conv1 if w is None else w).to(torch.float64)
    acc = torch.zeros(x.shape[0], 149, 149, 32, dtype=torch.float32)
    for ky, kx, ci in order:
        p = x[:, ky:ky + 297:2, kx:kx + 297:2, ci, None] * w[ky, kx, ci]
        if not fused:
            p = p.to(torch.float32).to(torch.float64)
        acc = (acc.to(torch.float64) + p).to(torch.float32)
    scale, shift = ow.affine["block1_conv1"]
    return XO.rn_bf16(relu(acc * scale + shift))


VARIANTS = {"kernel": {}, "reverse_order": dict(order=TAPS[::-1]), "unfused": dict(fused=False)}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_fp32_emulation_passes(sets, refs, ow, variant):
    """Not too tight: every input set, the kernel's arithmetic and two other correct fp32 evaluations"""
    singles = {}
    for name, t in sets.items():
        rep = XO.check(f"block1_conv1[{name}]", emulate(t, ow, **VARIANTS[variant]), refs[name], relu=True)
        print(f"{variant} {name}: single-valued {rep['single']:.4f}, max |y - z| / (E + half ulp) {rep['ratio']:.3f}")
        assert rep["n_fail"] == 0, XO.describe(rep)
        singles[name] = rep["single"]
    assert min(singles.values()) >= XO.SINGLE_FLOOR["block1_conv1_f32"], singles


def test_constant_tile_gives_relu_shift(sets, refs, ow):
    """the oracle standardises a constant tile to exact zeros: the accumulator is exactly 0, so every output is
    bf16(ReLU(shift)) and its interval holds that one value"""
    shift = ow.affine["block1_conv1"][1]
    want = XO.rn_bf16(torch.clamp_min(shift, 0.0))
    for i in (4, 5):
        assert not sets["oracle"][i].any()
        assert torch.equal(emulate(sets["oracle"][i:i + 1], ow)[0], want.expand(149, 149, 32))
        lo, hi = XO.interval(*(a[i] for a in refs["oracle"][1]), relu=True)
        assert torch.equal(lo, want.expand(149, 149, 32)) and torch.equal(hi, lo)
    assert np.abs(sets["oracle"][6]).max() > 500                           # the single-pixel tile's outlier


def _swap_30_31(y):
    return y[..., [*range(30), 31, 30]]


def _restandardize(t):
    """the kRaw branch on float input: (x - mean) * (1 / std) applied again, with the tile's own fp32 statistics"""
    x = torch.from_numpy(t).to(torch.float64).reshape(len(t), -1)
    m = x.mean(1)
    sd = torch.clamp_min(torch.sqrt(torch.clamp_min((x * x).mean(1) - m * m, 0.0)), 1 / np.sqrt(x.shape[1]))
    m, inv = m.to(torch.float32), (1 / sd).to(torch.float32)
    return ((torch.from_numpy(t) - m[:, None, None, None]) * inv[:, None, None, None]).numpy()


def _no_relu_on_5(y):
    return torch.cat([torch.clamp_min(y[..., :5], 0.0), y[..., 5:6], torch.clamp_min(y[..., 6:], 0.0)], -1)


def _zero_last_row(t):
    t = t.copy()
    t[:, 298] = 0
    return t


# name -> (tiles -> kernel input, emulate kwargs, output change, sets it must fail on, histogram condition)
MUTATIONS = {
    "taps_transposed": (None, dict(w="T"), None, ("oracle", "tf", "raw", "big"), None),
    "bgr": (lambda t: np.ascontiguousarray(t[..., ::-1]), {}, None, ("oracle", "tf", "raw", "big"), None),
    "last_row_zero": (_zero_last_row, {}, None, ("oracle", "tf", "raw", "big"), lambda h: set(h["row"]) == {148}),
    "channels_30_31_swapped": (None, {}, _swap_30_31, ("oracle", "tf", "raw", "big"),
                               lambda h: set(h["channel"]) <= {30, 31}),
    # a second standardisation only shows where the input is not already standardised
    "standardised_twice": (_restandardize, {}, None, ("raw", "big"), None),
    "relu_missing_on_5": (None, dict(relu=_no_relu_on_5), None, ("oracle", "tf", "raw", "big"),
                          lambda h: set(h["channel"]) == {5}),
}


@pytest.mark.parametrize("name", list(MUTATIONS))
def test_kernel_like_bugs_fail(sets, refs, ow, name):
    """Not too loose: each bug fails on every set it can show on, localised by the failure histogram"""
    pre, kw, post, must_fail, where = MUTATIONS[name]
    if kw.get("w") == "T":
        kw = dict(w=ow.conv1.permute(1, 0, 2, 3))                           # w[kx, ky] read for tap (ky, kx)
    for s in must_fail:
        t = sets[s] if pre is None else pre(sets[s])
        y = emulate(t, ow, **kw)
        if post is not None:
            y = post(y)
        rep = XO.check(f"block1_conv1[{s}]", y, refs[s], relu=True)
        print(name, XO.describe(rep))
        assert rep["n_fail"] > 0, (name, s)
        if where:
            hist = {k: list(v) for k, v in rep["hist"].items()}
            assert where(hist), (name, s, hist)
