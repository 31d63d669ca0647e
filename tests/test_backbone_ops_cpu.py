"""CPU tier: the per-op references and error bounds of oracle/xception_ops.py, checked without a GPU.

  * not too tight: an fp32 implementation with the kernels' rounding points but a different accumulation order (torch fp32
    conv / matmul) passes the check for every op of the plan, on one synthetic tile;
  * not too loose: kernel-like bugs (a depthwise tap off by 1 %, one corner tap missing at one pixel, the last 24-channel
    k-block dropped, a wrong BatchNorm shift on the last channel tile) fail it, and the failures point at the change;
  * wiring: the ops chained from the tile reproduce XceptionUQOracle(emulate_bf16=True) stage outputs.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import synth, xception_ops as XO, xception_uq as X


def _fp32_op(op, ins, ow, mutate=None):
    """fp32 implementation with the kernels' rounding points (accumulation order: torch's)"""
    f32 = torch.float32
    src = ins[op.inputs[0]]
    w_pw = ow.pw.get(op.layer)
    scale, shift = ow.affine.get(op.layer, (None, None))
    if mutate and mutate.get("layer") == op.layer:
        w_pw = mutate.get("pw", lambda w: w)(w_pw)
        shift = mutate.get("shift", lambda s: s)(shift)

    def epi(acc, res=None):
        y = acc * scale + shift
        if res is not None:
            y = y + res
        return XO.rn_bf16(torch.clamp_min(y, 0.0) if op.relu_out else y)

    def dw(x):
        d = ow.dw[op.layer]
        if mutate and mutate.get("layer") == op.layer and "dw" in mutate:
            return mutate["dw"](x, d, op.relu_in)
        x = torch.clamp_min(x, 0.0) if op.relu_in else x
        xp = F.pad(x, (0, 0, 1, 1, 1, 1))
        acc = torch.zeros_like(x)
        for k in range(9):
            acc = torch.addcmul(acc, xp[:, k // 3:k // 3 + x.shape[1], k % 3:k % 3 + x.shape[2], :], d[k // 3, k % 3])
        return XO.rn_bf16(acc)

    if op.kind == "conv1":
        mean, inv = X.XceptionUQOracle.tile_stats(src)
        m0 = torch.round(mean.double())
        x = torch.from_numpy(src).double().permute(0, 3, 1, 2) - m0[:, None, None, None]
        acc = F.conv2d(x.to(f32), ow.conv1.permute(3, 2, 0, 1), stride=2).permute(0, 2, 3, 1)
        s, h = (a.double() for a in ow.affine["block1_conv1"])
        g = inv.double()[:, None] * s
        hh = h - (mean.double() - m0)[:, None] * ow.conv1.double().sum((0, 1, 2)).float().double() * g
        y = (acc.double() * g.float().double()[:, None, None] + hh.float().double()[:, None, None]).float()
        return XO.rn_bf16(torch.clamp_min(y, 0.0))
    if op.kind == "conv2":
        w = ow.pw["block1_conv2"].reshape(64, 3, 3, 32).permute(0, 3, 1, 2)
        return epi(F.conv2d(src.permute(0, 3, 1, 2), w).permute(0, 2, 3, 1))
    if op.kind == "sub":
        return src[:, ::2, ::2, :].contiguous()
    if op.kind == "pooladd":
        return XO.pooladd_exact(src, ins[op.inputs[1]])
    if op.kind == "dw":
        return dw(src)
    res = ins[op.residual] if op.residual else None
    a = dw(src) if op.kind == "sep" else src
    return epi(a @ w_pw.T, res)


def chain(tile, ow, stop=None, mutate=None, sepmid=True):
    """all tagged outputs of one plan from uint8 tiles, each op computed by _fp32_op on the previous ops' outputs"""
    outs = {"tiles": tile}
    for op in XO.plan(sepmid):
        outs[op.tag] = _fp32_op(op, outs, ow, mutate)
        if op.tag == stop:
            break
    return outs


@pytest.fixture(scope="module")
def weights():
    return X.make_weights(seed=1)


@pytest.fixture(scope="module")
def ow(weights):
    return XO.OpWeights(weights)


@pytest.fixture(scope="module")
def tile():
    return synth.tiles_u8(1, seed=0, n_slides=1)


@pytest.fixture(scope="module")
def base(tile, ow):
    torch.set_num_threads(max(torch.get_num_threads(), 4))
    with torch.no_grad():
        return chain(tile, ow)


def _check(op, outs, ow):
    ins = {t: outs[t] for t in op.inputs}
    return XO.check(op.tag, outs[op.tag], XO.op_ref(op, ins, ow), relu=op.relu_out)


@pytest.mark.parametrize("sepmid", [True, False], ids=["sepmid", "unfused"])
def test_fp32_implementation_passes(base, tile, ow, sepmid):
    """Not too tight: every op of the plan, fp32 arithmetic in another order, on real intermediates"""
    outs = base if sepmid else chain(tile, ow, sepmid=False)
    with torch.no_grad():
        for op in XO.plan(sepmid):
            rep = _check(op, outs, ow)
            assert rep["n_fail"] == 0, XO.describe(rep)
            print(f"{op.tag} ({op.kind}): single-valued {rep['single']:.4f}, max |y - z| / E {rep['ratio']:.3f}")
            assert rep["single"] >= XO.single_floor(op), (op.tag, rep["single"])


def _fp32_head(h1, masks, ow, roll=0):
    """fp32 head with the kernels' rounding points (torch fp32 matmuls); `roll` != 0 applies the site-1 mask to the
    neighbouring activation (a mask on the wrong unit)"""
    inv_keep = float(np.float32(1.0) / (np.float32(1.0) - np.float32(0.1)))
    (W2, b2), W3, b3 = ow.hidden[1], ow.w3, ow.b3
    probs = []
    for t in range(masks.shape[1]):
        k1, k2 = (torch.from_numpy(masks[:, t, s]).float() for s in (0, 1))
        h2 = XO.rn_bf16(torch.clamp_min((h1 * torch.roll(k1, roll, 1)) @ W2.T * inv_keep + b2, 0.0))
        probs.append(torch.softmax((h2 * k2) @ W3 * inv_keep + b3, 1))
    p = torch.stack(probs)
    return p.mean(0), torch.sqrt(((p - p.mean(0)[None]) ** 2).mean(0))


def test_gap_and_head_fp32_pass(base, ow):
    """global average pool, hidden_0 as a GEMM op, and the fused head from that h1: fp32 implementations pass, the
    head's interval on the mean is narrow (<= 2e-3), and a mask applied to the neighbouring activation fails"""
    x = base["block14"]
    feats = x.double().mean((1, 2)).float()
    z, E = XO.gap_ref(x)
    assert ((feats.double() - z).abs() <= E).all()
    W1, b1 = ow.hidden[0]
    h1 = XO.rn_bf16(torch.clamp_min(XO.rn_bf16(feats) @ W1.T + b1, 0.0))
    rep = XO.check("hidden_0", h1, ("bound", XO.hidden0_ref(feats, ow)), relu=True)
    assert rep["n_fail"] == 0, XO.describe(rep)
    assert rep["single"] >= XO.SINGLE_FLOOR["hidden_0"], rep["single"]
    for T in (7, 32, 70):
        masks = X.keep_masks(1, T, 1024, 0.1, 77)
        h = XO.head_ref(h1, masks, ow)
        width = float((h["mean_hi"] - h["mean_lo"]).max())
        nm, ns, r = XO.check_head(*_fp32_head(h1, masks, ow), h)
        print(f"head T={T}: mean width {width:.2e}, std ratio {r:.3f}")
        assert nm == 0 and ns == 0
        assert width <= 2e-3
        nm, ns, _ = XO.check_head(*_fp32_head(h1, masks, ow, roll=1), h)
        assert nm > 0, f"T={T}: a mask on the wrong activation passes"


def test_wiring_matches_oracle_stages(base, tile, weights):
    """the per-op chain reproduces the bf16-emulated oracle's stage outputs (right weights, relu_in, residual source)"""
    st = {}
    with torch.no_grad():
        X.XceptionUQOracle(weights, emulate_bf16=True).backbone(tile, stages=st)
    for name, ref in st.items():
        got = base[name].numpy()
        d = np.abs(got - ref)
        assert d.max() <= 5e-2 * np.abs(ref).max() and d.mean() <= 2.5e-2 * np.abs(ref).mean(), name


def _mut_tap(x, d, relu_in):
    d = d.clone()
    d[2, 2] = XO.rn_bf16(d[2, 2] * 1.01)
    return XO.depthwise_exact(x, d, relu_in)


def _mut_corner(x, d, relu_in):
    y = XO.depthwise_exact(x, d, relu_in)
    d0 = d.clone()
    d0[0, 0] = 0
    y[:, 18, 18, :] = XO.depthwise_exact(x, d0, relu_in)[:, 18, 18, :]
    return y


def _mut_ktail(w):
    w = w.clone()
    w[:, 704:] = 0
    return w


def _mut_shift(s):
    s = s.clone()
    s[704:] += 0.05
    return s


MUTATIONS = {
    # a depthwise tap off by 1 % (tap (2, 2) of a middle-flow layer), in the fused sepconv and stand-alone
    "tap": ("block5_sepconv1", dict(dw=_mut_tap), None),
    "tap_unfused": ("block5_sepconv1_dw", dict(dw=_mut_tap), None),
    # one corner tap missing at one border pixel
    "corner": ("block5_sepconv1", dict(dw=_mut_corner), lambda h: set(h["row"]) == {18} and set(h["col"]) == {18}),
    # the partial last k-block (input channels 704..727) dropped
    "ktail": ("block8_sepconv2", dict(pw=_mut_ktail), None),
    # a wrong BatchNorm shift on the last channel tile of one GEMM
    "shift": ("block13_sepconv1", dict(shift=_mut_shift), lambda h: min(h["c//56"]) >= 12),
}


@pytest.mark.parametrize("name", list(MUTATIONS))
def test_kernel_like_bugs_fail(base, tile, ow, name):
    """Not too loose: each change fails the check of the op it is in, localised; the next op (fed the changed output)
    still passes, so a failure points at the op that is wrong"""
    tag, mut, where = MUTATIONS[name]
    sepmid = not tag.endswith("_dw") and not tag.startswith("block13")
    ops = XO.plan(sepmid)
    i = [op.tag for op in ops].index(tag)
    layer = ops[i].layer
    with torch.no_grad():
        outs = chain(tile, ow, stop=ops[i + 1].tag, mutate=dict(mut, layer=layer), sepmid=sepmid)
        rep = _check(ops[i], outs, ow)
        print(XO.describe(rep))
        assert rep["n_fail"] > 0
        if where:
            hist = {k: list(v) for k, v in rep["hist"].items()}
            assert where(hist), hist
        nxt = _check(ops[i + 1], outs, ow)
        assert nxt["n_fail"] == 0, XO.describe(nxt)
