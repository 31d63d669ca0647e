"""GPU tier: every op of the backbone plan checked alone, on its own GPU inputs, against a float64 reference with a
proven error bound (oracle/xception_ops.py).

For each tagged op, the inputs are the GPU's `debug_stage` outputs of the producing ops; the reference computes the op
in float64 and bounds what fp32 accumulation and the epilogue roundings of a correct kernel can change.  Every output
element must lie in [RN(act(z - E)), RN(act(z + E))]; depthwise, subsample and max-pool + add must match exactly.  A
failure prints the failing elements and where they cluster (image, row, column, channel block, work-item position).

Both plans are walked: the default one (fused middle-flow `sepconv_mid_kernel`) and BQ_SEPMID=off (stand-alone depthwise
+ pointwise GEMM).  8 tiles fill max_batch = 8, so the middle-flow work items of 160 padded rows cross image boundaries;
the first 3 tiles alone (a partial micro-batch) must give bit-identical outputs.
"""
import os

import numpy as np
import pytest
import torch

from helpers import degenerate_tiles
from oracle import synth, xception_ops as XO, xception_uq as X

pytestmark = pytest.mark.gpu

PLANS = {"sepmid": XO.plan(True), "unfused": XO.plan(False)}


@pytest.fixture(scope="module")
def weights():
    return X.make_weights(seed=1)


@pytest.fixture(scope="module")
def tiles():
    """4 synthetic tiles + 4 degenerate ones (large uniform regions, all-zero channels deep in the net) = max_batch"""
    return np.ascontiguousarray(np.concatenate([synth.tiles_u8(4, seed=0, n_slides=3), degenerate_tiles()]))


@pytest.fixture(scope="module")
def opw(weights):
    return XO.OpWeights(weights, device="cuda")


@pytest.fixture(scope="module")
def ifaces(weights):
    """one interface per plan; BQ_SEPMID is read when the model is created"""
    from biscuit_b200.uq import UncertaintyInterface
    out = {}
    old = os.environ.get("BQ_SEPMID")
    try:
        for name, mode in (("sepmid", "on"), ("unfused", "off")):
            os.environ["BQ_SEPMID"] = mode
            out[name] = UncertaintyInterface(weights, max_batch=8)
    finally:
        if old is None:
            os.environ.pop("BQ_SEPMID", None)
        else:
            os.environ["BQ_SEPMID"] = old
    yield out
    for it in out.values():
        it.close()


@pytest.fixture(scope="module")
def stage_cache():
    return {}


def stage(ifaces, cache, tiles, plan, tag):
    key = (plan, tag)
    if key not in cache:
        cache[key] = ifaces[plan].debug_stage(tiles, tag)
    return cache[key]


CASES = [(p, op) for p, ops in PLANS.items() for op in ops]


@pytest.mark.parametrize("plan,op", CASES, ids=[f"{p}-{op.tag}" for p, op in CASES])
def test_op_within_bound(ifaces, stage_cache, tiles, opw, plan, op):
    y = stage(ifaces, stage_cache, tiles, plan, op.tag)
    ins = {t: (tiles if t == "tiles" else torch.from_numpy(stage(ifaces, stage_cache, tiles, plan, t)).cuda())
           for t in op.inputs}
    rep = XO.check(op.tag, torch.from_numpy(y).cuda(), XO.op_ref(op, ins, opw), relu=op.relu_out)
    print(f"{plan} {op.tag} ({op.kind}): single-valued {rep['single']:.4f}, max |y - z| / E {rep['ratio']:.3f}")
    assert rep["n_fail"] == 0, XO.describe(rep)
    assert rep["single"] >= XO.single_floor(op), (op.tag, rep["single"])
    # a partial micro-batch gives the same bits as the same tiles in the full one
    y3 = ifaces[plan].debug_stage(tiles[:3], op.tag)
    diff = np.nonzero((y3 != y[:3]).reshape(3, -1).any(1))[0]
    assert y3.tobytes() == y[:3].tobytes(), f"{op.tag}: tiles {diff} differ between 3- and 8-tile micro-batches"


def test_plans_cover_every_tag(ifaces, tiles):
    """the listing in oracle/xception_ops.py is the library's plan, tag for tag and in order, for both plans; the two
    plans differ only in the middle flow (blocks 5-12)"""
    for plan, ops in PLANS.items():
        assert ifaces[plan].debug_tags() == [op.tag for op in ops], plan
    mid = lambda tag: any(tag == f"block{b}" or tag.startswith(f"block{b}_") for b in range(5, 13))   # noqa: E731
    assert [op.tag for op in PLANS["sepmid"] if not mid(op.tag)] == [op.tag for op in PLANS["unfused"] if not mid(op.tag)]
    with pytest.raises(Exception):
        ifaces["sepmid"].debug_stage(tiles[:1], "block5_sepconv1_dw")     # fused: no stand-alone depthwise
    with pytest.raises(Exception):
        ifaces["sepmid"].debug_stage(tiles[:1], "dw0")


@pytest.mark.parametrize("plan", list(PLANS))
def test_global_average_pool_within_bound(ifaces, stage_cache, tiles, plan):
    x = torch.from_numpy(stage(ifaces, stage_cache, tiles, plan, "block14")).cuda()
    _, _, feats = ifaces[plan].predict(tiles, T=2, seed=1, return_features=True)
    z, E = XO.gap_ref(x)
    d = (torch.from_numpy(feats).cuda().to(torch.float64) - z).abs()
    print(f"{plan} gap: max |y - z| / E {float((d / E).max()):.3f}")
    bad = torch.nonzero(d > E)
    assert len(bad) == 0, f"{len(bad)} features outside the bound, first (tile, c): {bad[:8].tolist()}"


@pytest.mark.parametrize("t_samples", [7, 32, 70])
def test_head_within_bound(ifaces, tiles, opw, t_samples):
    """hidden_0 as a GEMM op on bf16(features), then the fused MC-dropout head from the GPU's own h1 with injected masks:
    T < 32, T == 32, T > 32 (Chan merge).  The interval on the mean is narrow enough (<= 2e-3) that a mask applied to
    the neighbouring activation, which moves the mean by ~5e-3 to 2e-2, fails (tests/test_backbone_ops_cpu.py)."""
    it = ifaces["sepmid"]
    masks = X.keep_masks(len(tiles), t_samples, 1024, 0.1, 77)
    mean, std, feats = it.predict(tiles, T=t_samples, masks=masks, return_features=True)
    h1 = torch.from_numpy(it.debug_h1(len(tiles))).cuda()
    rep = XO.check("hidden_0", h1, ("bound", XO.hidden0_ref(torch.from_numpy(feats).cuda(), opw)), relu=True)
    print(f"hidden_0: single-valued {rep['single']:.4f}, max |y - z| / E {rep['ratio']:.3f}")
    assert rep["n_fail"] == 0, XO.describe(rep)
    assert rep["single"] >= XO.SINGLE_FLOOR["hidden_0"], rep["single"]
    h = XO.head_ref(h1, masks, opw)
    nm, ns, r = XO.check_head(mean, std, h)
    width = float((h["mean_hi"] - h["mean_lo"]).max())
    print(f"head T={t_samples}: mean interval width <= {width:.2e}, max |d std| / allowed {r:.3f}")
    assert nm == 0 and ns == 0, (nm, ns, mean, h["mean_lo"].cpu().numpy(), h["mean_hi"].cpu().numpy())
    assert width <= 2e-3
