"""CPU tier: the general MC-dropout head reference (oracle/xception_ops.py: head_ref, hidden0_ref) checked without a GPU,
over a matrix of hidden widths, class counts, dropout placements, rates and sample counts.

  * not too tight: an fp32 emulation of mc_head_fused_kernel (hidden_1 accumulated per K = 16 MMA in issue order, the
    epilogue, the fma chain into the prelogits, the fp32 softmax, per-chunk shuffle statistics and Chan's merge) passes
    everywhere, and so does an fp32 implementation that sums in another order (torch matmuls, one two-pass mean / std);
  * not too loose: kernel-like bugs fail, and only in the configurations they affect;
  * sharp: the interval on the mean is at most 2e-3 wide for rates <= 0.5.
"""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import xception_ops as XO, xception_uq as X

f32, f64 = torch.float32, torch.float64
N_TILES = 2


def _f32(x):
    return x.to(f32)


def head_weights(W, C, seed):
    """hidden_1 and prelogits as the head holds them (bf16 W2 [out, in], fp32 b2, W3 [W, C], b3), with the scales of
    weights.random_init; hidden_0 [W, 2048] for the site-0 check"""
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, dtype=f64)                  # noqa: E731
    W1 = XO.rn_bf16((rn(W, 2048) * 0.27 / np.sqrt(2048)).to(f32))
    W2 = XO.rn_bf16((rn(W, W) * np.sqrt(2.0) / np.sqrt(W)).to(f32))
    return SimpleNamespace(device="cpu", hidden=[(W1, (rn(W) * 0.05).to(f32)), (W2, (rn(W) * 0.05).to(f32))],
                           w3=(rn(W, C) / np.sqrt(W)).to(f32), b3=(rn(C) * 0.05).to(f32))


def make_h1(n, T, W, per_sample, seed):
    """bf16 post-ReLU activations with about half of the units at 0, like hidden_0's"""
    g = torch.Generator().manual_seed(1000 + seed)
    shape = (n, T, W) if per_sample else (n, W)
    return XO.rn_bf16(torch.clamp_min(torch.randn(*shape, generator=g), 0.0) * 1.5)


def make_masks(n, T, W, rate, sites, seed):
    enabled = [i for i, on in enumerate(sites) if on]
    return X.keep_masks(n, T, 2048 if sites[0] else W, rate, seed, sites=enabled)


def _site_masks(masks, sites, W):
    """per-site float keep-masks [n, T, W] (all ones behind a disabled site)"""
    slot = {s: i for i, s in enumerate(s for s, on in enumerate(sites) if on)}
    n, T = masks.shape[:2]
    ones = torch.ones(n, T, W)
    return {s: (torch.from_numpy(masks[:, :, slot[s], :W]).float() if s in slot else ones) for s in (1, 2)}


def emulate(h1, masks, ow, rate, sites, mut=None, kernel_order=True):
    """fp32 emulation of mc_head_fused_kernel -> (mean, std) [n, C] float32.  kernel_order=False sums in another order:
    torch fp32 matmuls for hidden_1 and the prelogits, torch's softmax, one two-pass mean / std over all T."""
    mut = mut or ()
    (W2, b2), W3, b3 = ow.hidden[1], ow.w3, ow.b3
    W, C = W2.shape[0], W3.shape[1]
    n, T = masks.shape[:2]
    ik = XO.inv_keep(rate)
    ik1 = ik if (sites[1] or "inv_keep_disabled" in mut) else 1.0
    ik2 = ik if (sites[2] or "inv_keep_disabled" in mut) else 1.0
    km = _site_masks(masks, sites, W)
    k1, k2 = km[1], km[2]
    if "site2_counter" in mut and sites[1] and sites[2]:
        k2 = k1                                       # site 2 drawn with site 1's Philox counter: site 1's keep pattern
    a = (h1 if h1.dim() == 3 else h1[:, None, :].expand(n, T, W)) * k1          # [n, T, W]: an exact selection
    a = a.reshape(n * T, W)
    if kernel_order:
        acc = torch.zeros(n * T, W, dtype=f32)
        for g in range(W // XO.MMA_K):                # one MMA per K = 16 in issue order: 16 exact products, then + acc
            s = slice(g * XO.MMA_K, (g + 1) * XO.MMA_K)
            acc = _f32(acc.double() + _f32(a[:, s].double() @ W2[:, s].double().T).double())
    else:
        acc = a @ W2.T
    if "skip_second_block" in mut:                    # the second 256-column MMA block of each 512-column half
        for h0 in range(0, W, 512):
            acc[:, h0 + 256:h0 + 512] = 0.0
    x = _f32(_f32(acc * np.float32(ik1)) + b2)
    h2 = XO.rn_bf16(torch.clamp_min(x, 0.0)) * k2.reshape(n * T, W)
    w3 = W3.reshape(C, W).T if "w3_transposed" in mut else W3       # [W][C] read as [C][W]
    if kernel_order:
        logit = torch.zeros(n * T, C, dtype=f32)
        for j in range(W):                            # fmaf(x, w3[j][c], logit[c]), units ascending
            logit = _f32(h2[:, j:j + 1].double() * w3[j].double() + logit.double())
    else:
        logit = h2 @ w3
    z = _f32(logit * np.float32(ik2)) + b3
    if "softmax_all_slots" in mut:                    # all 8 logit slots (unused ones 0) enter the softmax
        z = torch.cat([z, torch.zeros(n * T, 8 - C)], 1)
    if kernel_order:
        e = torch.exp(z - z.max(1, keepdim=True).values)
        den = torch.zeros(n * T, dtype=f32)
        for c in range(z.shape[1]):
            den = den + e[:, c]
        p = (e / den[:, None])[:, :C]
    else:
        p = torch.softmax(z, 1)[:, :C]
    p = p.reshape(n, T, C)
    if not kernel_order:
        m = p.mean(1)
        return m, torch.sqrt(((p - m[:, None]) ** 2).mean(1))
    return _chunk_stats(p, drop_partial="drop_partial_chunk" in mut)


def _butterfly(v):
    """warp xor-shuffle sum over the 32 lanes (dim 1), fp32"""
    for o in (16, 8, 4, 2, 1):
        v = v + v[:, torch.arange(32) ^ o]
    return v[:, 0]


def _chunk_stats(p, drop_partial=False):
    n, T, C = p.shape
    r_n = 0.0
    r_mean, r_m2 = torch.zeros(n, C), torch.zeros(n, C)
    for sc in range((T + 31) // 32):
        cnt = min(32, T - 32 * sc)
        if drop_partial and cnt < 32:
            continue
        v = torch.zeros(n, 32, C)
        v[:, :cnt] = p[:, 32 * sc:32 * sc + cnt]
        cn = np.float32(cnt)
        cm = _butterfly(v) / cn
        d = v - cm[:, None]
        d[:, cnt:] = 0.0
        m2 = _butterfly(d * d)
        if r_n == 0.0:
            r_mean, r_m2 = cm, m2
        else:
            tot = np.float32(r_n + cn)
            delta = cm - r_mean
            r_mean = r_mean + delta * cn / tot
            r_m2 = r_m2 + (m2 + delta * delta * np.float32(r_n) * cn / tot)
        r_n += cnt
    return r_mean, torch.sqrt(r_m2 / np.float32(r_n))


DEFAULT = (False, True, True)
# (W, C, sites, rate, T)
CONFIGS = [
    (64, 8, DEFAULT, 0.1, 33),
    (128, 2, (True, False, True), 0.9, 33),
    (192, 3, (False, True, False), 0.1, 7),
    (256, 8, (True, True, True), 0.1, 32),
    (320, 5, DEFAULT, 0.5, 64),
    (576, 2, (False, False, True), 0.1, 33),
    (576, 8, (True, True, False), 0.1, 40),
    (1024, 3, DEFAULT, 0.1, 70),
    (1024, 2, (True, False, False), 0.0, 32),
]
IDS = [f"W{w}-C{c}-s{''.join('1' if x else '0' for x in s)}-p{r}-T{t}" for w, c, s, r, t in CONFIGS]


@pytest.fixture(scope="module")
def cases():
    torch.set_num_threads(max(torch.get_num_threads(), 4))
    out = {}
    with torch.no_grad():
        for i, (W, C, sites, rate, T) in enumerate(CONFIGS):
            ow = head_weights(W, C, seed=i)
            h1 = make_h1(N_TILES, T, W, sites[0], seed=i)
            masks = make_masks(N_TILES, T, W, rate, sites, seed=50 + i)
            out[IDS[i]] = (ow, h1, masks, rate, sites, XO.head_ref(h1, masks, ow, rate, sites))
    return out


@pytest.mark.parametrize("cid", IDS)
@pytest.mark.parametrize("kernel_order", [True, False], ids=["kernel_order", "other_order"])
def test_fp32_head_passes(cases, cid, kernel_order):
    """Not too tight: both fp32 implementations lie within the bound; the check stays sharp"""
    ow, h1, masks, rate, sites, h = cases[cid]
    with torch.no_grad():
        rep = XO.head_report(*emulate(h1, masks, ow, rate, sites, kernel_order=kernel_order), h)
    print(f"{cid}: mean width {rep['width']:.2e}, |d mean| / half-width {rep['ratio_mean']:.3f}, "
          f"|d std| / allowed {rep['ratio_std']:.3f}")
    assert rep["n_fail_mean"] == 0 and rep["n_fail_std"] == 0, XO.describe_head(cid, rep)
    if rate <= 0.5:
        assert rep["width"] <= 2e-3, rep["width"]


# mutation -> the configurations it affects (W, C, sites, rate, T)
MUTATIONS = {
    "w3_transposed": lambda W, C, s, r, T: True,
    "softmax_all_slots": lambda W, C, s, r, T: C < 8,
    "drop_partial_chunk": lambda W, C, s, r, T: T % 32 != 0,
    "site2_counter": lambda W, C, s, r, T: s[1] and s[2],
    "inv_keep_disabled": lambda W, C, s, r, T: r > 0 and not (s[1] and s[2]),
    "skip_second_block": lambda W, C, s, r, T: any(min(512, W - h0) > 256 for h0 in range(0, W, 512)),
}


@pytest.mark.parametrize("mut", list(MUTATIONS))
def test_kernel_like_bugs_fail_where_they_apply(cases, mut):
    """Not too loose: each change fails the check in every configuration it affects, and in no other"""
    failed = {}
    with torch.no_grad():
        for cid, (ow, h1, masks, rate, sites, h) in cases.items():
            rep = XO.head_report(*emulate(h1, masks, ow, rate, sites, mut=(mut,)), h)
            failed[cid] = rep["n_fail_mean"] + rep["n_fail_std"] > 0
            if failed[cid]:
                print(XO.describe_head(f"{mut} {cid}", rep).splitlines()[0])
    expected = {cid: bool(MUTATIONS[mut](*cfg)) for cid, cfg in zip(IDS, CONFIGS)}
    assert failed == expected, {cid: (failed[cid], expected[cid]) for cid in IDS if failed[cid] != expected[cid]}


def _box_differences(zlo, zhi):
    """differences z_j - z_c [.., c, j] of logits bounded one by one"""
    return zlo[..., None, :] - zhi[..., :, None], zhi[..., None, :] - zlo[..., :, None]


def test_softmax_interval_is_sigmoid_for_two_classes():
    """for C = 2 the softmax bound is the sigmoid of the logit difference at its two ends"""
    g = torch.Generator().manual_seed(3)
    zlo = torch.randn(64, 2, generator=g, dtype=f64)
    zhi = zlo + torch.rand(64, 2, generator=g, dtype=f64) * 0.1
    plo, phi = XO.softmax_interval(*_box_differences(zlo, zhi))
    assert torch.allclose(plo[:, 1], torch.sigmoid(zlo[:, 1] - zhi[:, 0]), rtol=0, atol=1e-15)
    assert torch.allclose(phi[:, 0], torch.sigmoid(zhi[:, 0] - zlo[:, 1]), rtol=0, atol=1e-15)
    # the exact softmax of any point of the box lies inside, for 8 classes
    zlo8 = torch.randn(256, 8, generator=g, dtype=f64) * 3
    zhi8 = zlo8 + torch.rand(256, 8, generator=g, dtype=f64)
    plo8, phi8 = XO.softmax_interval(*_box_differences(zlo8, zhi8))
    for _ in range(8):
        p = torch.softmax(zlo8 + torch.rand(256, 8, generator=g, dtype=f64) * (zhi8 - zlo8), 1)
        assert ((p >= plo8 - 1e-15) & (p <= phi8 + 1e-15)).all()


def test_logit_differences_contain_every_activation_choice():
    """logit_diff_interval: for h2 anywhere in [h2lo, h2hi], the fp32 logits (fma chain, * ik2, + b3) of that h2 have
    differences inside the interval, and the interval is narrower than the one of logits bounded one by one"""
    g = torch.Generator().manual_seed(4)
    W, C, ik2 = 256, 8, XO.inv_keep(0.1)
    w3 = (torch.randn(W, C, generator=g, dtype=f64) / 16).float().double()
    b3 = torch.randn(C, generator=g, dtype=f64) * 0.05
    lo = XO.rn_bf16(torch.clamp_min(torch.randn(16, W, generator=g), 0.0)).double()
    hi = torch.where(torch.rand(16, W, generator=g) < 0.2, XO.rn_bf16(lo.float() * (1 + 2 ** -7)).double(), lo)
    dlo, dhi = XO.logit_diff_interval(lo, hi, w3, b3, ik2)
    for _ in range(8):
        h2 = torch.where(torch.rand(16, W, generator=g) < 0.5, lo, hi)
        logit = torch.zeros(16, C, dtype=f32)
        for j in range(W):
            logit = _f32(h2[:, j:j + 1] * w3[j].float().double() + logit.double())
        z = (_f32(logit * np.float32(ik2)) + b3.float()).double()
        d = z[:, None, :] - z[:, :, None]
        assert ((d >= dlo) & (d <= dhi)).all()
    err, llo, lhi = XO._fma_chain_error(lo, hi, w3)
    zlo, zhi = llo * ik2 + b3, lhi * ik2 + b3
    blo, bhi = _box_differences(zlo, zhi)
    assert ((dhi - dlo) <= (bhi - blo) + 1e-12).all() and float((dhi - dlo).mean()) < float((bhi - blo).mean())


def test_slack_grows_with_chunks():
    """the statistics allowance follows the number of Chan merges: none for T <= 32, 127 at T = 4096"""
    _, e1, eta1 = XO.head_slack(32, 2)
    _, e2, eta2 = XO.head_slack(33, 2)
    _, e3, eta3 = XO.head_slack(4096, 8)
    assert len(eta1) == 0 and len(eta2) == 1 and len(eta3) == 127
    assert e1 < e2 < e3 and e3 < 1e-4


def test_hidden0_per_sample_passes_and_mask_shift_fails():
    """site 0: hidden_0 per sample on bf16(features) * keep0 with the GEMM's alpha = 1/(1-p) epilogue.  An fp32 GEMM in
    another order passes; a site-0 mask applied to the neighbouring feature fails"""
    W, T, rate = 128, 5, 0.1
    ow = head_weights(W, 2, seed=7)
    g = torch.Generator().manual_seed(8)
    feats = torch.clamp_min(torch.randn(N_TILES, 2048, generator=g), 0.0)
    k0 = X.keep_masks(N_TILES, T, 2048, rate, 9, sites=[0])[:, :, 0]
    W1, b1 = ow.hidden[0]

    def fp32_h1(shift=0):
        a = XO.rn_bf16(feats)[:, None, :] * torch.roll(torch.from_numpy(k0).float(), shift, 2)
        return XO.rn_bf16(torch.clamp_min(_f32(a @ W1.T * np.float32(XO.inv_keep(rate))) + b1, 0.0))

    z, E = XO.hidden0_ref(feats, ow, k0=k0, rate=rate)
    assert tuple(z.shape) == (N_TILES, T, W)
    ref = ("bound", (z.reshape(-1, W), E.reshape(-1, W)))                 # rows in (tile, sample) order
    rep = XO.check("hidden_0", fp32_h1().reshape(-1, W), ref, relu=True)
    assert rep["n_fail"] == 0, XO.describe(rep)
    assert rep["single"] >= XO.SINGLE_FLOOR["hidden_0"], rep["single"]
    assert XO.check("hidden_0", fp32_h1(shift=1).reshape(-1, W), ref, relu=True)["n_fail"] > 0


def test_rejected_configurations():
    """a model without any dropout site and an interface with `uq` off are refused, not silently run as another model"""
    from biscuit_b200.hp import nature2022
    from biscuit_b200.uq import UncertaintyInterface
    with pytest.raises(ValueError, match="at least one"):
        nature2022.replace(dropout_sites=(False, False, False)).dropout_site_mask
    for sites in ALL_SITE_MASKS:
        assert nature2022.replace(dropout_sites=sites).dropout_site_mask == sum(1 << i for i, on in enumerate(sites) if on)
    with pytest.raises(ValueError, match="uq"):
        UncertaintyInterface({}, config=nature2022.replace(uq=False))


ALL_SITE_MASKS = [tuple(bool(m >> i & 1) for i in range(3)) for m in range(1, 8)]
