"""TEST INFRASTRUCTURE ONLY -- one-op references of the Xception-UQ backbone and head, with proven error bounds.

Each op of the CUDA execution plan (biscuit_b200/csrc/model.cu: `build_plan`) is checked ALONE, on the inputs the GPU
itself produced for it (`UncertaintyInterface.debug_stage` of the producing ops).  A reference returns, per output element,
the exact value `z` (float64) and a bound `E` on how far a correct kernel's fp32 arithmetic can move it.  The check is

    RN(act(z - E)) <= y <= RN(act(z + E))

with RN = round to the output type (fp32 -> bf16 for activations) and act = the op's ReLU or the identity.  Both are
monotone, so the check needs no ulp allowance; it is element by element, not against a tensor-wide maximum.

Rounding points are taken from the kernels, not from oracle/xception_uq.py:
  * depthwise (dwpipe_sm100.cuh, and the producers of sepconv2d_sm100.cuh / sepmid_sm100.cuh): acc = 0, then the nine
    taps top row first, left to right, acc = fp32(acc + x * w); x and w are bf16, so each product is exact in fp32 and
    the fma is an ordinary add.  Then RN to bf16.  Emulated exactly: the check is equality.
  * GEMM epilogues (gemm_sm100.cuh, sepconv2d / sepmid): fp32 accumulator, then RN(acc * scale), RN(+ shift),
    RN(+ residual), ReLU, RN to bf16.  The accumulator of a K-term tensor-core dot product is bounded by
    K * 2^-23 * sum|a||w|: 2^-23 rather than fp32's unit roundoff 2^-24 allows for accumulation that truncates.
  * max-pool + add, subsample (layers.cuh): exact.
  * block1_conv1 (conv1_sm100.cuh): conv(W, x - m0) over W = hi + mid + lo on the tensor cores, then one fp32 FMA
    with the per-tile constants g = scale / sd and h = shift - (m - m0) * sum(W) * g.  On float tiles the caller already
    standardised (conv1_kernel<float>, layers.cuh): 27 fp32 fmas from 0 in (ky, kx, ci) order, then the GEMM epilogue.
  * global average pool (layers.cuh): an n-term fp32 sum and one division.
  * MC-dropout head (gemm hidden_0 + head_sm100.cuh): intervals through the two bf16 activations h1, h2 and the fp32
    prelogits, the softmax bounded through its monotonicity in each logit, then the fp32 allowances of the per-chunk
    statistics and their Chan merge (head_slack), for every class count, width, dropout placement and rate.

All functions take torch tensors (float32 holding bf16 values, NHWC) and work on the tensors' device.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from oracle.xception_arch import ENTRY_BLOCKS, MIDDLE_BLOCKS

U = 2.0 ** -24        # unit roundoff of fp32 round-to-nearest
UA = 2.0 ** -23       # per-term bound of a tensor-core fp32 accumulation (allows truncation)
TINY = 2.0 ** -126    # absolute slack per fp32 step (flushed subnormals)
BN_EPS = np.float32(1e-3)


def rn_bf16(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16, round to nearest even, returned as float32"""
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float32)


# ------------------------------------------------------------------------------------------------------------------
# weights in the form the kernels hold them (model.cu: load_bn / load_conv_gemm / load_sep / load_dense)
# ------------------------------------------------------------------------------------------------------------------
def _bf16_np(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).to(torch.float32)


def bn_affine(w, bn):
    """fp32 scale / shift exactly as load_bn computes them: s = g / sqrtf(v + eps), shift = b - m * s"""
    g, b = np.float32(w[f"{bn}/gamma"]), np.float32(w[f"{bn}/beta"])
    m, v = np.float32(w[f"{bn}/moving_mean"]), np.float32(w[f"{bn}/moving_variance"])
    s = (g / np.sqrt(v + BN_EPS)).astype(np.float32)
    ms = (m * s).astype(np.float32)
    return torch.from_numpy(s), torch.from_numpy((b - ms).astype(np.float32))


class OpWeights:
    """Per-layer kernel-side weights: `dw[name]` bf16 [3, 3, C]; `pw[name]` bf16 [N, K] (K tap-major for 3x3);
    `affine[name]` fp32 (scale, shift); block1_conv1 kept in fp32 [3, 3, 3, 32]; head kernels as the head holds them."""

    def __init__(self, weights: dict, device="cpu"):
        self.device = device
        t = lambda a: a.to(device)                                           # noqa: E731
        self.dw, self.pw, self.affine = {}, {}, {}
        from oracle.xception_arch import layer_table
        for kind, name, cin, cout in layer_table():
            if kind.startswith("conv3x3"):
                k = np.asarray(weights[f"{name}/kernel"], np.float32)         # HWIO
                if name == "block1_conv1":
                    self.conv1 = t(torch.from_numpy(np.ascontiguousarray(k)))
                else:
                    self.pw[name] = t(_bf16_np(k.reshape(-1, k.shape[-1]).T))  # [N, tap * cin + c]
                self.affine[name] = tuple(t(a) for a in bn_affine(weights, f"{name}_bn"))
            elif kind == "res":
                k = np.asarray(weights[f"{name}/kernel"], np.float32)
                self.pw[name] = t(_bf16_np(k.reshape(-1, k.shape[-1]).T))
                self.affine[name] = tuple(t(a) for a in bn_affine(weights, f"{name}_bn"))
            else:
                d = np.asarray(weights[f"{name}/depthwise_kernel"], np.float32)[:, :, :, 0]
                self.dw[name] = t(_bf16_np(d))
                p = np.asarray(weights[f"{name}/pointwise_kernel"], np.float32)[0, 0]
                self.pw[name] = t(_bf16_np(p.T))
                self.affine[name] = tuple(t(a) for a in bn_affine(weights, f"{name}_bn"))
        HeadWeights.__init__(self, weights, device)


class HeadWeights:
    """The head's kernel-side weights alone: `hidden[i]` = (bf16 [out, in], fp32 bias) of hidden_0 / hidden_1,
    `w3` fp32 [W, C] and `b3` fp32 [C] of the prelogits"""

    def __init__(self, weights: dict, device="cpu"):
        self.device = device
        t = lambda a: a.to(device)                                           # noqa: E731
        self.hidden = [(t(_bf16_np(np.asarray(weights[f"hidden_{i}/kernel"]).T)),
                        t(torch.from_numpy(np.asarray(weights[f"hidden_{i}/bias"], np.float32))))
                       for i in range(2)]
        self.w3 = t(torch.from_numpy(np.asarray(weights["prelogits/kernel"], np.float32)))
        self.b3 = t(torch.from_numpy(np.asarray(weights["prelogits/bias"], np.float32)))


# ------------------------------------------------------------------------------------------------------------------
# the plan: one entry per tagged op (model.cu: build_plan), in execution order
# ------------------------------------------------------------------------------------------------------------------
class Op:
    """kind: conv1 | conv2 | sub | res | sep (fused depthwise + pointwise) | dw | pw | pooladd.
    `inputs`: the tags whose outputs feed the op ('tiles' = the uint8 tiles, or float32 tiles the caller standardised);
    `layer`: weight name."""

    def __init__(self, tag, kind, inputs, layer=None, relu_in=False, relu_out=False, residual=None):
        self.tag, self.kind, self.inputs, self.layer = tag, kind, list(inputs), layer
        self.relu_in, self.relu_out, self.residual = relu_in, relu_out, residual

    def __repr__(self):
        return f"Op({self.tag}, {self.kind})"


def plan(sepmid: bool = True):
    """The tagged ops of the default plan (sepmid=True: fused middle flow) or of BQ_SEPMID=off"""
    ops = [Op("block1_conv1", "conv1", ["tiles"], "block1_conv1", relu_out=True),
           Op("block1_conv2", "conv2", ["block1_conv1"], "block1_conv2", relu_out=True)]
    x = "block1_conv2"

    def sep(b, i, src, relu_in, relu_out, fused, residual=None, tag=None):
        name = f"block{b}_sepconv{i}"
        tag = tag or name
        if fused:
            ops.append(Op(tag, "sep", [src] + ([residual] if residual else []), name, relu_in, relu_out, residual))
        else:
            ops.append(Op(f"{name}_dw", "dw", [src], name, relu_in))
            ops.append(Op(tag, "pw", [f"{name}_dw"] + ([residual] if residual else []), name, False, relu_out, residual))
        return tag

    def res_block(b, x, relu_first, fused):
        ops.append(Op(f"block{b}_sub", "sub", [x]))
        ops.append(Op(f"block{b}_res", "res", [f"block{b}_sub"], f"block{b}_res"))
        y = sep(b, 1, x, relu_first, True, fused)
        y = sep(b, 2, y, False, False, fused)
        ops.append(Op(f"block{b}", "pooladd", [y, f"block{b}_res"]))
        return f"block{b}"

    for b, _, _ in ENTRY_BLOCKS:
        x = res_block(b, x, b != 2, fused=b in (2, 3))
    for b in MIDDLE_BLOCKS:
        y = sep(b, 1, x, True, True, sepmid)
        y = sep(b, 2, y, False, True, sepmid)
        x = sep(b, 3, y, False, False, sepmid, residual=x, tag=f"block{b}")
    x = res_block(13, x, True, fused=False)
    y = sep(14, 1, x, False, True, False)
    sep(14, 2, y, False, True, False, tag="block14")
    return ops


# Non-vacuity: per op, the share of output elements whose bf16 interval holds exactly one value must not fall below
# these floors (exact ops -- subsample, depthwise, max-pool + add -- are 1 by construction).  Each floor is 0.85 x the
# share a CPU run of tests/test_backbone_ops_cpu.py found on one synthetic tile, rounded down, the smaller of the two
# plans; a bound that widened for one op would show here.  The K * 2^-23 accumulation bound is what makes the
# intervals of the 728- and 1024-deep GEMMs wider (block13_res: K = 728 with little cancellation).
# "block1_conv1_f32" is block1_conv1 on float tiles (conv1_f32_ref): 0.85 x 0.9914, the smallest share over the four
# input sets of tests/test_input_route_gpu.py (the +-1e4 set) measured on a B200.
SINGLE_FLOOR = {
    "hidden_0": 0.4, "block1_conv1_f32": 0.84,
    "block1_conv1": 0.82, "block1_conv2": 0.75, "block2_res": 0.81, "block2_sepconv1": 0.83, "block2_sepconv2": 0.77,
    "block3_res": 0.74, "block3_sepconv1": 0.8, "block3_sepconv2": 0.69, "block4_res": 0.62, "block4_sepconv1": 0.76,
    "block4_sepconv2": 0.36, "block5_sepconv1": 0.6, "block5_sepconv2": 0.61, "block5": 0.5, "block6_sepconv1": 0.6,
    "block6_sepconv2": 0.61, "block6": 0.51, "block7_sepconv1": 0.58, "block7_sepconv2": 0.59, "block7": 0.52,
    "block8_sepconv1": 0.6, "block8_sepconv2": 0.6, "block8": 0.53, "block9_sepconv1": 0.6, "block9_sepconv2": 0.6,
    "block9": 0.53, "block10_sepconv1": 0.59, "block10_sepconv2": 0.6, "block10": 0.53, "block11_sepconv1": 0.6,
    "block11_sepconv2": 0.6, "block11": 0.53, "block12_sepconv1": 0.6, "block12_sepconv2": 0.62, "block12": 0.51,
    "block13_res": 0.22, "block13_sepconv1": 0.6, "block13_sepconv2": 0.37, "block14_sepconv1": 0.48, "block14": 0.46,
}


def single_floor(op):
    return SINGLE_FLOOR[op.tag] if op.kind not in ("sub", "dw", "pooladd") else 1.0


# ------------------------------------------------------------------------------------------------------------------
# references: (z, E) per output element
# ------------------------------------------------------------------------------------------------------------------
def depthwise_exact(x: torch.Tensor, dw: torch.Tensor, relu_in: bool) -> torch.Tensor:
    """bit-exact depthwise 3x3 'same' of the kernels: fp32 acc from 0, taps in row-major order, then RN to bf16"""
    x = x.to(torch.float32)
    if relu_in:
        x = torch.clamp_min(x, 0.0)
    n, h, w, c = x.shape
    xp = F.pad(x, (0, 0, 1, 1, 1, 1))
    acc = torch.zeros_like(x)
    for ky in range(3):
        for kx in range(3):
            acc = acc + xp[:, ky:ky + h, kx:kx + w, :] * dw[ky, kx].to(torch.float32)
    return rn_bf16(acc)


def epilogue_bound(z, E, scale=None, shift=None, residual=None):
    """fp32 epilogue steps RN(* scale), RN(+ shift), RN(+ residual) applied to an interval z +- E (float64)"""
    if scale is not None:
        s = scale.to(torch.float64)
        z, E = z * s, E * s.abs()
        E = E + U * (z.abs() + E) + TINY
    if shift is not None:
        z = z + shift.to(torch.float64)
        E = E + U * (z.abs() + E) + TINY
    if residual is not None:
        z = z + residual.to(torch.float64)
        E = E + U * (z.abs() + E) + TINY
    return z, E


def gemm_ref(a: torch.Tensor, w: torch.Tensor, scale, shift, residual=None):
    """a [..., K] bf16 values, w [N, K] bf16 values -> (z, E) [..., N]"""
    a64, w64 = a.to(torch.float64), w.to(torch.float64)
    z = a64 @ w64.T
    E = a.shape[-1] * UA * (a64.abs() @ w64.abs().T)
    return epilogue_bound(z, E, scale, shift, residual)


def conv2_ref(x: torch.Tensor, ow: OpWeights):
    """block1_conv2: 3x3 valid implicit GEMM, K = 288 (tap-major)"""
    w = ow.pw["block1_conv2"].to(torch.float64).reshape(64, 3, 3, 32).permute(0, 3, 1, 2)     # OIHW
    x64 = x.to(torch.float64).permute(0, 3, 1, 2)
    z = F.conv2d(x64, w).permute(0, 2, 3, 1)
    E = 288 * UA * F.conv2d(x64.abs(), w.abs()).permute(0, 2, 3, 1)
    return epilogue_bound(z, E, *ow.affine["block1_conv2"])


def conv1_ref(tiles_u8: np.ndarray, ow: OpWeights):
    """block1_conv1 (conv1_tc_kernel): z = BN(conv(W, (x - m) * inv)) with the fp32 m / inv of tile_stats_kernel."""
    from oracle.xception_uq import XceptionUQOracle
    dev = ow.device
    mean, inv = XceptionUQOracle.tile_stats(tiles_u8)                     # fp32, as tile_stats_kernel rounds them
    mf, isf = mean.to(torch.float64).to(dev), inv.to(torch.float64).to(dev)
    m0 = torch.round(mf)                                                  # rint: half to even, like torch.round
    W = ow.conv1.to(torch.float64).permute(3, 2, 0, 1)                    # [32, 3, 3, 3] OIHW
    scale, shift = (a.to(torch.float64) for a in ow.affine["block1_conv1"])
    x = torch.from_numpy(tiles_u8).to(dev).to(torch.float64).permute(0, 3, 1, 2)
    xs = (x - mf[:, None, None, None]) * isf[:, None, None, None]
    z = F.conv2d(xs, W, stride=2).permute(0, 2, 3, 1) * scale + shift
    xm = x - m0[:, None, None, None]
    A = F.conv2d(xm, W, stride=2).permute(0, 2, 3, 1)                     # the accumulator's exact value
    S = F.conv2d(xm.abs(), W.abs(), stride=2).permute(0, 2, 3, 1)
    sumw = W.sum((1, 2, 3))
    g = isf[:, None] * scale[None]                                        # exact (two fp32 factors)
    d = (mf - m0)[:, None]
    h = shift[None] - d * sumw[None] * g
    g32 = g.to(torch.float32).to(torch.float64)
    # 96 products (hi | mid | lo thirds of W, 27 taps padded to 32) in one fp32 accumulator
    e_acc = 96 * UA * S
    e_g = (A.abs() + e_acc) * (g32 - g).abs()[:, None, None] + e_acc * g32.abs()[:, None, None]
    e_h = (U * h.abs() + (d * g).abs() * (U * sumw.abs() + 64 * 2.0 ** -53 * W.abs().sum((1, 2, 3)))[None]
           + 8 * 2.0 ** -53 * (shift.abs()[None] + (d * sumw[None] * g).abs()))
    E = e_g + e_h[:, None, None] + TINY
    E = E + U * (z.abs() + E) + TINY                                      # the FMA's rounding
    return z, E


def gamma(k: int, u: float = U) -> float:
    """gamma_k = k u / (1 - k u): the relative error bound of a k-step RN recurrence (Higham, Accuracy and Stability, 3.1)"""
    return k * u / (1 - k * u)


def conv1_f32_ref(tiles_f32, ow: OpWeights):
    """block1_conv1 on float tiles the caller already standardised (conv1_kernel<float>, layers.cuh): z = BN(conv(W, x))
    in float64 from the caller's fp32 values x and the fp32 weights W [3, 3, 3, 32] (3x3, stride 2, valid).

    Rounding points of the kernel, per output and channel:
      * acc = 0, then 27 fp32 fmas acc = RN(x * w + acc) in (ky, kx, ci) order.  Each step rounds once, relative error
        <= u on the partial sum, so |acc - A| <= gamma_27 * S with A = sum x w and S = sum |x| |w| (Higham 3.1; the
        bound holds for any summation order, so it does not rely on the order).  Subnormal partial sums add at most
        2^-150 per step, covered by TINY.  The float64 conv that gives A is itself off by <= gamma_27(2^-53) * S, which
        is added to the same E so that z is not taken as exact.
      * RN(acc * scale), RN(+ shift): epilogue_bound.
      * ReLU and RN to bf16: interval (both monotone).
    tiles_f32: float32 NHWC [n, 299, 299, 3] (numpy or torch) -> (z, E) [n, 149, 149, 32] float64 on ow.device"""
    dev = ow.device
    x = torch.as_tensor(np.asarray(tiles_f32) if not torch.is_tensor(tiles_f32) else tiles_f32)
    assert x.dtype == torch.float32, x.dtype
    x = x.to(dev).to(torch.float64).permute(0, 3, 1, 2)
    W = ow.conv1.to(torch.float64).permute(3, 2, 0, 1)                    # [32, 3, 3, 3] OIHW
    A = F.conv2d(x, W, stride=2).permute(0, 2, 3, 1)
    S = F.conv2d(x.abs(), W.abs(), stride=2).permute(0, 2, 3, 1)
    E = (gamma(27) + gamma(27, 2.0 ** -53)) * S + 27 * TINY
    return epilogue_bound(A, E, *ow.affine["block1_conv1"])


def pooladd_exact(y: torch.Tensor, res: torch.Tensor) -> torch.Tensor:
    """MaxPool 3x3 s2 'same' (-inf padding) + residual: RN_bf16(fp32(max) + fp32(res))"""
    from oracle.xception_uq import _same_pad_s2
    t = y.to(torch.float32).permute(0, 3, 1, 2)
    pt, pb = _same_pad_s2(t.shape[2])
    pl, pr = _same_pad_s2(t.shape[3])
    m = F.max_pool2d(F.pad(t, (pl, pr, pt, pb), value=float("-inf")), 3, 2).permute(0, 2, 3, 1)
    return rn_bf16(m + res.to(torch.float32))


def subsample_exact(x: torch.Tensor) -> torch.Tensor:
    return x[:, ::2, ::2, :]


def gap_ref(x: torch.Tensor):
    """features (fp32) = fp32 sum over the map in order, / HW  -> (z, E) with the n-term sum bound"""
    n, h, w, c = x.shape
    hw = h * w
    x64 = x.to(torch.float64).reshape(n, hw, c)
    z = x64.mean(1)
    E = (hw + 1) * U * x64.abs().sum(1) / hw
    E = E + U * (z.abs() + E) + TINY
    return z, E


def op_ref(op: Op, ins: dict, ow: OpWeights):
    """-> ('exact', y_ref) or ('bound', (z, E)) for one plan op, from its input tensors `ins` (tag -> tensor)"""
    src = ins[op.inputs[0]]
    if op.kind == "conv1":
        f32 = str(src.dtype).replace("torch.", "") == "float32"            # tiles the caller standardised
        return "bound", conv1_f32_ref(src, ow) if f32 else conv1_ref(src, ow)
    if op.kind == "conv2":
        return "bound", conv2_ref(src, ow)
    if op.kind == "sub":
        return "exact", subsample_exact(src)
    if op.kind == "dw":
        return "exact", depthwise_exact(src, ow.dw[op.layer], op.relu_in)
    if op.kind == "pooladd":
        return "exact", pooladd_exact(src, ins[op.inputs[1]])
    res = ins[op.residual] if op.residual else None
    if op.kind == "res":
        return "bound", gemm_ref(src, ow.pw[op.layer], *ow.affine[op.layer])
    if op.kind == "pw":
        return "bound", gemm_ref(src, ow.pw[op.layer], *ow.affine[op.layer], residual=res)
    if op.kind == "sep":
        d = depthwise_exact(src, ow.dw[op.layer], op.relu_in)
        return "bound", gemm_ref(d, ow.pw[op.layer], *ow.affine[op.layer], residual=res)
    raise ValueError(op.kind)


# ------------------------------------------------------------------------------------------------------------------
# the check and its report
# ------------------------------------------------------------------------------------------------------------------
def interval(z, E, relu):
    """bf16 interval [RN(act(z - E)), RN(act(z + E))] (fp64 -> fp32 -> bf16: a composition of monotone roundings)"""
    lo, hi = z - E, z + E
    if relu:
        lo, hi = torch.clamp_min(lo, 0.0), torch.clamp_min(hi, 0.0)
    return rn_bf16(lo.to(torch.float32)), rn_bf16(hi.to(torch.float32))


def where(bad: torch.Tensor, shape):
    """failing NHWC coordinates and histograms over image, row, column, channel, channel block and work-item position"""
    idx = torch.nonzero(bad.reshape(shape)).cpu().numpy()
    n, h, w, c = shape
    i, y, x, ch = idx.T if len(idx) else (np.zeros(0, int),) * 4
    flat = (i * h + y) * w + x
    keys = {"image": i, "row": y, "col": x, "channel": ch, "c//64": ch // 64, "c//56": ch // 56,
            "last n-block(64)": ch >= (c - 1) // 64 * 64, "gemm row%128": flat % 128}
    if (h, w) == (19, 19):
        keys["sepmid padded row%160"] = ((i * 20 + y) * 20 + x) % 160
    else:
        keys["sep2d y%8"], keys["sep2d x%16"] = y % 8, x % 16
    hist = {}
    for k, v in keys.items():
        vals, cnt = np.unique(v, return_counts=True)
        order = np.argsort(-cnt)[:8]
        hist[k] = {int(vals[j]): int(cnt[j]) for j in order}
    return [tuple(int(t) for t in r) for r in idx[:8]], hist


def check(tag, y: torch.Tensor, ref, relu=False):
    """y: GPU output (float32 holding bf16), ref: op_ref result -> report dict (n_fail, where, non-vacuity, max |y-z|/E)"""
    kind, val = ref
    y = y.to(val[0].device if kind == "bound" else val.device).to(torch.float32)
    if kind == "exact":
        assert tuple(y.shape) == tuple(val.shape), (tag, tuple(y.shape), tuple(val.shape))
        bad = y != val                                                     # -0 == +0
        single, ratio = 1.0, 0.0
    else:
        z, E = val
        assert tuple(y.shape) == tuple(z.shape), (tag, tuple(y.shape), tuple(z.shape))
        lo, hi = interval(z, E, relu)
        bad = (y < lo) | (y > hi) | torch.isnan(y)
        single = float((lo == hi).to(torch.float64).mean())
        # distance from the exact value in units of the bound plus half a bf16 ulp of the output (<= 1 when contained)
        zz = torch.clamp_min(z, 0.0) if relu else z
        half_ulp = torch.ldexp(torch.ones_like(y, dtype=torch.float64), torch.frexp(y).exponent.to(torch.int64) - 9)
        ratio = float(((y.to(torch.float64) - zz).abs() / (E + half_ulp)).max())
    n_bad = int(bad.sum())
    rep = dict(tag=tag, n=int(y.numel()), n_fail=n_bad, single=single, ratio=ratio)
    if n_bad:
        shape = tuple(y.shape) if y.dim() == 4 else (y.shape[0], 1, 1, y.shape[-1])
        rep["first"], rep["hist"] = where(bad, shape)
    return rep


def describe(rep):
    s = f"{rep['tag']}: {rep['n_fail']} of {rep['n']} elements outside the bound"
    if rep["n_fail"]:
        s += f"; first (tile, y, x, c): {rep['first']}"
        for k, v in rep["hist"].items():
            s += f"\n    {k}: {v}"
    return s


# ------------------------------------------------------------------------------------------------------------------
# head: hidden_0 is an ordinary GEMM op (checked with gemm_ref); the fused head kernel runs from the GPU's own h1
# ------------------------------------------------------------------------------------------------------------------
MMA_K = 16            # K of one tcgen05.mma (bf16): the head's hidden_1 accumulates 1024 / 16 of them in k order


def inv_keep(rate: float) -> float:
    """the kernels' fp32 1/(1-p)"""
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(rate)))


def hidden0_ref(features: torch.Tensor, ow: OpWeights, k0=None, rate: float = 0.0):
    """hidden_0 on bf16(features) [n, 2048]: GEMM epilogue RN(acc * alpha) + b1, ReLU, bf16 -> (z, E) [n, W].
    With dropout on the pooled features (site 0), k0 = the site-0 keep-masks [n, T, 2048]: mc_expand_kernel writes one
    row bf16(features) * keep0 per (tile, sample) (an exact selection) and the GEMM runs on those n * T rows with
    alpha = 1/(1-p) (prepare_head) -> (z, E) [n, T, W]."""
    a = rn_bf16(features)
    W1, b1 = ow.hidden[0]
    if k0 is None:
        return gemm_ref(a, W1, None, b1)                                  # alpha = 1: RN(acc * 1) is exact
    k0 = torch.as_tensor(k0).to(a.device, torch.float32)
    alpha = torch.tensor(inv_keep(rate), dtype=torch.float64, device=a.device)
    return gemm_ref(a[:, None, :] * k0, W1, alpha, b1)


def mma_chain_bound(a: torch.Tensor, w: torch.Tensor):
    """(z, E) of a @ w.T accumulated as the head kernel issues it: one fp32 accumulator that the K / 16 MMA instructions
    update in k order (dependent MMAs on one accumulator execute in issue order).  Each instruction adds 16 exact
    products to the accumulator; bounded as a 17-term sum in any order with truncation: 17 * 2^-23 * (sum of the 16
    |products| + |accumulator before it|).  This is the K * 2^-23 bound of gemm_ref applied per instruction, and it
    does not grow with K the way that bound does."""
    n, k = a.shape
    g = k // MMA_K
    a64, w64 = a.to(torch.float64).reshape(n, g, MMA_K), w.to(torch.float64).reshape(w.shape[0], g, MMA_K)
    part = torch.einsum("ngk,ogk->ngo", a64, w64)                        # [n, groups, out]
    S = a.to(torch.float64).abs() @ w.to(torch.float64).abs().T
    P = torch.cumsum(part, 1)
    z = P[:, -1]
    E = 17 * UA * (S + P[:, :-1].abs().sum(1))
    return z, E * (1 + 2 * g * 17 * UA)                                 # the accumulator's own error, carried along


def _fma_chain_error(lo, hi, w):
    """bound on the rounding error of the sequential fp32 fma chain over units j (ascending) of x_j * w[j, c], for any x
    in [lo, hi] (>= 0): one rounding of each partial sum, u * sum_j max |partial sum j| -> [n, C]"""
    wp, wn = torch.clamp_min(w, 0.0), torch.clamp_max(w, 0.0)
    tlo, thi = lo[:, :, None] * wp + hi[:, :, None] * wn, hi[:, :, None] * wp + lo[:, :, None] * wn   # [n, units, C]
    plo, phi = torch.cumsum(tlo, 1), torch.cumsum(thi, 1)
    return U * torch.maximum(plo.abs(), phi.abs()).sum(1) + TINY * w.shape[0], plo[:, -1], phi[:, -1]


def _round_interval(lo, hi, mul, add):
    """fp32 RN(RN(x * mul) + add) over [lo, hi] (mul > 0) -> float64 interval"""
    lo, hi = lo * mul, hi * mul
    lo, hi = lo - U * lo.abs() - TINY, hi + U * hi.abs() + TINY
    lo, hi = lo + add, hi + add
    return lo - U * lo.abs() - TINY, hi + U * hi.abs() + TINY


def logit_diff_interval(h2lo, h2hi, w3, b3, ik2):
    """Interval of the fp32 logit differences z_j - z_c, z = RN(RN(l * ik2) + b3) with l the fp32 fma chain over the
    bf16 activations h2 in [h2lo, h2hi] (>= 0) -> (dlo, dhi) [n, c, j].

    Every logit is a function of the same h2, so the difference is bounded through the weights w3[:, j] - w3[:, c]
    (bounding each logit alone and subtracting the ends would count each h2 unit's uncertainty twice): its exact part
    lies in ik2 * [sum_k min, sum_k max of h2_k (w3[k, j] - w3[k, c])] + b3_j - b3_c.  Each logit adds its own fp32
    error: the fma chain's (_fma_chain_error), scaled by ik2, then u |l ik2| and u |z| of the two roundings."""
    C = w3.shape[1]
    err, llo, lhi = _fma_chain_error(h2lo, h2hi, w3)
    a = ik2 * (torch.maximum(llo.abs(), lhi.abs()) + err)                    # >= |RN(l) * ik2|
    eps = ik2 * err + U * a + U * (a * (1 + U) + b3.abs()) + 3 * TINY         # [n, C]: |z~ - (ik2 l + b3)|
    dw = (w3[:, None, :] - w3[:, :, None]).reshape(w3.shape[0], C * C)       # [units, (c, j)]
    dp, dn = torch.clamp_min(dw, 0.0), torch.clamp_max(dw, 0.0)
    dlo = (h2lo @ dp + h2hi @ dn).reshape(-1, C, C)
    dhi = (h2hi @ dp + h2lo @ dn).reshape(-1, C, C)
    db = b3[None, :] - b3[:, None]                                           # [c, j]: b3_j - b3_c
    e = eps[:, None, :] + eps[:, :, None]
    return ik2 * dlo + db - e, ik2 * dhi + db + e


def softmax_interval(dlo, dhi):
    """softmax p_c = 1 / (1 + sum_{j != c} exp(z_j - z_c)) falls with every difference d[c, j] = z_j - z_c, so for
    differences in [dlo, dhi] ([..., c, j]): p_c in [1 / (1 + sum_{j != c} exp(dhi[c, j])), 1 / (1 + sum_{j != c}
    exp(dlo[c, j]))] (C = 2: the sigmoid of the logit difference at its two ends)"""
    C = dlo.shape[-1]
    off = ~torch.eye(C, dtype=torch.bool, device=dlo.device)
    return 1.0 / (1.0 + (torch.exp(dhi) * off).sum(-1)), 1.0 / (1.0 + (torch.exp(dlo) * off).sum(-1))


CHUNK = 32            # samples per chunk of the head kernel's statistics (one per lane of a row warp)


def head_slack(T: int, C: int):
    """-> (dp, e_mean, eta): the fp32 rounding allowances of the head's softmax and statistics (head_sm100.cuh), for T
    samples in K = ceil(T / 32) chunks and C classes; u = 2^-24, probabilities are <= 1.

      * softmax (per sample): t_c = RN(z_c - max) is off by u |t_c|, which exp turns into a relative error u |t_c| on
        e_c; expf adds <= 2 ulp (4u relative); the C-term fp32 sum of the denominator (>= 1: its largest term is
        exp(0)) adds (C - 1) u; the division u.  With p_c |t_c| <= e^-|t_c| |t_c| <= 1/e and sum_j p_j |t_j| <= (C-1)/e,
        |RN(p_c) - p_c| <= u (1/e + 4 + 4 + (C-1) + (C-1)/e + 1) + O(u^2) <= dp = (12 + 2 C) u.
      * chunk mean: a 5-level shuffle butterfly over 32 lanes (invalid lanes add 0) and one division: |cm~ - cm| <=
        gamma_6 max|p| <= 6u (+ O(u^2)).
      * Chan merge k of r_mean: delta = RN(cm - r_mean), RN(delta * cn), RN(/ tot), RN(r_mean + .): the new exact mean
        is a convex combination of the old one and cm, so the carried error stays <= max(E_{k-1}, 6u), and the three
        roundings of the increment (|delta| <= 1) plus the one of the sum (|r_mean| <= 1) add 4u:
        E_mean <= e_mean = (6 + 4 (K - 1)) u.
      * M2: the chunk M2 uses d = RN(p - cm~) with cm~ = cm + eps: sum (d_j - eps)^2 = M2_chunk + cn eps^2 exactly (the
        d_j of the exact chunk mean sum to 0), then the square and the butterfly: a relative gamma_7 on nonnegative
        terms.  The merge term RN(RN(RN(delta^2) * r_n) * cn) / tot) has delta off by eta_k <= E_{k-1} + 6u + u R
        (R: the range of the tile's probabilities, which bounds |delta|), so it moves by <= min(na, nb) (2 R eta_k +
        eta_k^2) with min(na, nb) <= cn_k; its four roundings and the two additions into r_m2 are relative errors on
        nonnegative terms, gamma_(2K + 12) overall with the final RN(r_m2 / r_n).
      * std = sqrtf(var): |sqrt(a) - sqrt(b)| <= min(sqrt(|a - b|), |a - b| / sqrt(b)), and sqrtf's own rounding u.
    Returns dp, e_mean and eta [K - 1] (eta_k, k = 1..K-1), each with a 2^-10 relative margin for the O(u^2) terms."""
    K = (T + CHUNK - 1) // CHUNK
    g = 1 + 2.0 ** -10
    dp = (12 + 2 * C) * U * g
    e_mean = (6 + 4 * (K - 1)) * U * g
    eta = np.array([(13 + 4 * (k - 1)) * U * g for k in range(1, K)])
    return dp, e_mean, eta


def head_ref(h1: torch.Tensor, masks, ow, rate: float = 0.1, sites=(False, True, True), rows_per_block: int = 4096):
    """Fused MC-dropout head (head_sm100.cuh) from the GPU's own hidden_0 output and injected keep-masks.

    h1: bf16 values [n, W], or [n, T, W] when site 0 is on (hidden_0 is then per sample); masks: uint8 [n, T, n_sites,
    mask_w] with the enabled sites in ascending order (mask_w = 2048 with site 0 on, else W); W and C are read from the
    weights (`ow.hidden[1]`, `ow.w3`, `ow.b3`).  A disabled site has no mask and a scale of 1, as in the kernel
    (`slot < 0`, `inv_keep1` / `inv_keep2`).

    Per sample: the masked operand (exact), hidden_1 as the kernel's chain of K = 16 MMAs (mma_chain_bound), RN(* 1/(1-p)
    or 1), RN(+ b2), ReLU and bf16 at both interval ends, the site-2 mask, the fp32 fma chain into the C prelogits,
    RN(* 1/(1-p) or 1), RN(+ b3) bounded as logit differences (logit_diff_interval), then the softmax bound
    (softmax_interval).  The statistics are then checked with the
    fp32 allowances of head_slack.
    -> dict with, per [n, C]: mean_lo / mean_hi (the GPU mean must lie inside), std_z / std_allow (|std - std_z| <=
    std_allow); plo / phi [n, T, C] per sample, and T, K, the slack terms."""
    dev = ow.device
    f64 = torch.float64
    W2, b2 = ow.hidden[1][0], ow.hidden[1][1].to(f64)
    W3, b3 = ow.w3.to(f64), ow.b3.to(f64)
    W, C = W2.shape[0], W3.shape[1]
    masks = torch.as_tensor(masks).to(dev)
    n, T = masks.shape[:2]
    slot, k = {}, 0
    for i, on in enumerate(sites):
        if on:
            slot[i], k = k, k + 1
    assert masks.shape[2] == k, (tuple(masks.shape), sites)
    ik = inv_keep(rate)
    ik1, ik2 = (ik if sites[1] else 1.0), (ik if sites[2] else 1.0)
    h1 = torch.as_tensor(h1).to(dev, f64)
    per_sample = h1.dim() == 3
    assert per_sample == bool(sites[0]), "hidden_0 is per sample exactly when site 0 is on"
    tb = max(1, rows_per_block // n)
    plo_b, phi_b = [], []
    for t0 in range(0, T, tb):
        t1 = min(T, t0 + tb)
        a = h1[:, t0:t1] if per_sample else h1[:, None, :].expand(n, t1 - t0, W)
        if 1 in slot:
            a = a * masks[:, t0:t1, slot[1], :W].to(f64)                  # the masked operand: an exact selection
        z2, E2 = mma_chain_bound(a.reshape(-1, W), W2)
        h2lo, h2hi = _round_interval(z2 - E2, z2 + E2, ik1, b2)
        h2lo = rn_bf16(torch.clamp_min(h2lo, 0.0).to(torch.float32)).to(f64)
        h2hi = rn_bf16(torch.clamp_min(h2hi, 0.0).to(torch.float32)).to(f64)
        if 2 in slot:
            k2 = masks[:, t0:t1, slot[2], :W].reshape(-1, W).to(f64)
            h2lo, h2hi = h2lo * k2, h2hi * k2
        plo, phi = softmax_interval(*logit_diff_interval(h2lo, h2hi, W3, b3, ik2))
        plo_b.append(plo.reshape(n, t1 - t0, C))
        phi_b.append(phi.reshape(n, t1 - t0, C))
    plo, phi = torch.cat(plo_b, 1), torch.cat(phi_b, 1)                  # [n, T, C]
    dp, e_mean, eta = head_slack(T, C)
    K = (T + CHUNK - 1) // CHUNK
    pz = 0.5 * (plo + phi)
    std_z = pz.std(1, unbiased=False)
    # population std is 1-Lipschitz in the max norm: it moves by at most the largest change of one sample
    lip = torch.maximum(phi - pz, pz - plo).amax(1) + dp
    R = phi.amax(1) - plo.amin(1) + 2 * dp
    cn = [min(CHUNK, T - CHUNK * k) for k in range(1, K)]
    d_m2 = T * (7 * U) ** 2 + sum(c * (2 * R * e + e * e) for c, e in zip(cn, eta)) * (1 + 8 * U)
    s_hi = std_z + lip
    s_lo = torch.clamp_min(std_z - lip, 0.0)
    d_var = d_m2 / T + s_hi ** 2 * (2 * K + 12) * U * (1 + 2.0 ** -10)
    d_std = torch.minimum(torch.sqrt(d_var), d_var / s_lo) + 2 * U * s_hi + TINY
    return dict(mean_lo=plo.mean(1) - dp - e_mean, mean_hi=phi.mean(1) + dp + e_mean, std_z=std_z,
                std_allow=lip + d_std, plo=plo, phi=phi, T=T, K=K, dp=dp, e_mean=e_mean)


def head_report(mean, std, h):
    """GPU mean / std [n, C] against head_ref's result -> report dict: n_fail_mean, n_fail_std, width (the widest mean
    interval), ratio_mean (max |mean - mid| / half-width), ratio_std (max |std - std_z| / allowed), and on a failure the
    first failing (tile, class) with their intervals"""
    dev = h["mean_lo"].device
    mean = torch.as_tensor(np.asarray(mean)).to(dev, torch.float64)
    std = torch.as_tensor(np.asarray(std)).to(dev, torch.float64)
    lo, hi = h["mean_lo"], h["mean_hi"]
    mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
    bad_m = (mean < lo) | (mean > hi) | torch.isnan(mean)
    ds = (std - h["std_z"]).abs()
    bad_s = (ds > h["std_allow"]) | torch.isnan(std)
    rep = dict(n=int(mean.numel()), n_fail_mean=int(bad_m.sum()), n_fail_std=int(bad_s.sum()),
               width=float((hi - lo).max()), ratio_mean=float(((mean - mid).abs() / half).max()),
               ratio_std=float((ds / h["std_allow"]).max()), T=h["T"], K=h["K"], first=[])
    for i, c in torch.nonzero(bad_m | bad_s)[:8].tolist():
        rep["first"].append(dict(tile=i, cls=c, group=i // 4, quadrant=i % 4, mean=float(mean[i, c]),
                                 mean_interval=(float(lo[i, c]), float(hi[i, c])), std=float(std[i, c]),
                                 std_z=float(h["std_z"][i, c]), std_allow=float(h["std_allow"][i, c])))
    return rep


def check_head(mean, std, h):
    """-> (n_fail_mean, n_fail_std, max |d std| / allowed); head_report has the details"""
    rep = head_report(mean, std, h)
    return rep["n_fail_mean"], rep["n_fail_std"], rep["ratio_std"]


def describe_head(tag, rep):
    """one line per failing (tile, class): the tile's four-tile group and TMEM quadrant, the value and its interval"""
    s = (f"{tag}: {rep['n_fail_mean']} means and {rep['n_fail_std']} stds of {rep['n']} outside the bound "
         f"(T = {rep['T']}, {rep['K']} sample chunks of 32)")
    for f in rep["first"]:
        s += (f"\n    tile {f['tile']} (group {f['group']}, quadrant {f['quadrant']}) class {f['cls']}: mean {f['mean']:.7f}"
              f" in [{f['mean_interval'][0]:.7f}, {f['mean_interval'][1]:.7f}]?  std {f['std']:.7f} vs {f['std_z']:.7f}"
              f" +- {f['std_allow']:.2e}")
    return s
