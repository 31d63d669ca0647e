"""GPU tier: Xception-UQ MC-dropout inference (CUDA, through the C ABI) against the CPU oracle
(oracle/xception_uq.py -- restated from Slideflow/Keras, parity with TensorFlow itself unpinned).

Tolerances (stated per north_star):
  * vs the bf16-emulated oracle (same rounding points as the CUDA path, fp32 accumulation in a
    different order, re-rounded to bf16 after each of the 36 layers so 1-ulp flips compound):
    backbone stages  max|d| <= 5e-2 * max|ref|,  mean|d| <= 2.5e-2 * mean|ref|
    (measured on B200: 0.2% after block1, 1.3% after block14);
    per-tile mean / std with INJECTED dropout masks: |d| <= 4e-3 absolute;
  * vs the fp32 oracle (the reference's arithmetic type): mean / std |d| <= 1.5e-2 absolute;
  * independently sampled masks: statistical tolerance 6 * std / sqrt(T) on the mean.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import synth, xception_uq as X

pytestmark = pytest.mark.gpu

N_TILES = 6
T = 30
SEED = 1234


@pytest.fixture(scope="module")
def weights():
    return X.make_weights(seed=1)


@pytest.fixture(scope="module")
def tiles():
    return synth.tiles_u8(N_TILES, seed=0, n_slides=3)


@pytest.fixture(scope="module")
def iface(weights):
    from biscuit_b200.uq import UncertaintyInterface
    return UncertaintyInterface(weights, max_batch=4)     # < N_TILES: exercises a partial micro-batch


@pytest.fixture(scope="module")
def oracle_bf16(weights, tiles):
    o = X.XceptionUQOracle(weights, emulate_bf16=True)
    stages = {}
    import torch
    with torch.no_grad():
        feats = o.backbone(tiles, stages=stages)
    return o, stages, feats


STAGES = ["block1_conv1", "block1_conv2", "block2", "block3", "block4", "block5", "block8", "block12",
          "block13", "block14"]


@pytest.mark.parametrize("stage", STAGES)
def test_backbone_stage_parity(iface, tiles, oracle_bf16, stage):
    _, stages, _ = oracle_bf16
    got = iface.debug_stage(tiles[:4], stage)
    ref = stages[stage][:4]
    assert got.shape == ref.shape, (got.shape, ref.shape)
    d = np.abs(got - ref)
    stats = dict(max_d=float(d.max()), max_ref=float(np.abs(ref).max()), mean_d=float(d.mean()),
                 mean_ref=float(np.abs(ref).mean()))
    print(stage, stats)
    assert d.max() <= 5e-2 * np.abs(ref).max(), stats
    assert d.mean() <= 2.5e-2 * np.abs(ref).mean(), stats


def test_entry_conv_on_degenerate_tiles(weights):
    """block1_conv1 runs on the tensor cores with the standardisation moved behind the convolution (conv1_sm100.cuh).
    That is only safe if the convolution never carries a large common term: constant tiles (blank background: std = 0,
    so 1 / max(std, 1/sqrt(N)) = 518), near-constant tiles, black / white tiles and a high-contrast checkerboard must
    match the oracle (which standardises first, in fp32) to bf16 rounding -- at most one bf16 ulp, on few outputs."""
    import torch
    from biscuit_b200.uq import UncertaintyInterface
    rng = np.random.default_rng(5)
    t = np.zeros((8, 299, 299, 3), np.uint8)
    t[0] = 255                                            # white background
    t[1] = 0                                              # black
    t[2] = 237                                            # constant, odd value
    t[3] = 200; t[3, 150, 150, 1] = 201                   # a single pixel differs: std = 0.0019
    t[4] = 128 + (rng.random((299, 299, 3)) < 0.02)       # sparse +1 noise
    t[5] = (np.indices((299, 299)).sum(0) % 2 * 255).astype(np.uint8)[..., None]   # checkerboard 0 / 255
    t[6] = rng.integers(0, 256, (299, 299, 3), dtype=np.uint8)
    t[7] = rng.integers(250, 256, (299, 299, 3), dtype=np.uint8)                   # bright, low contrast
    it = UncertaintyInterface(weights, max_batch=8)
    got = it.debug_stage(t, "block1_conv1")
    o = X.XceptionUQOracle(weights, emulate_bf16=True)
    stages = {}
    with torch.no_grad():
        o.backbone(t, stages=stages)
    ref = stages["block1_conv1"]
    assert got.shape == ref.shape
    for i in range(len(t)):
        d = np.abs(got[i] - ref[i])
        # one bf16 ulp is <= 2^-7 relative; the absolute floor covers outputs that sit on the ReLU boundary
        # (pre-activations of +-1e-6 land on 0 on one side and on a tiny positive number on the other)
        ulp = np.maximum(np.maximum(np.abs(ref[i]), np.abs(got[i])) * 2.0 ** -7, 1e-5)
        bad = d > ulp * 1.01
        assert not bad.any(), (i, float(d.max()), float(np.abs(ref[i]).max()), int(bad.sum()))
        assert (d > 0).mean() <= 0.02, (i, float((d > 0).mean()))          # and only a few outputs differ at all
    it.close()


def test_features_and_uq_with_injected_masks(iface, tiles, oracle_bf16, weights):
    o, _, feats_ref = oracle_bf16
    masks = X.keep_masks(N_TILES, T, 1024, 0.1, SEED)
    mean, std, feats = iface.predict(tiles, T=T, masks=masks, return_features=True)
    fr = feats_ref.numpy()
    assert np.abs(feats - fr).max() <= 3e-2 * np.abs(fr).max()
    m_ref, s_ref = o.predict_uq(tiles, T=T, masks=masks)
    print("bf16-tier  d_mean", np.abs(mean - m_ref).max(), "d_std", np.abs(std - s_ref).max())
    assert np.abs(mean - m_ref).max() <= 4e-3
    assert np.abs(std - s_ref).max() <= 4e-3
    assert np.allclose(mean.sum(1), 1.0, atol=1e-5)
    # fp32 oracle = the reference's arithmetic type
    o32 = X.XceptionUQOracle(weights, emulate_bf16=False)
    m32, s32 = o32.predict_uq(tiles, T=T, masks=masks)
    print("fp32-tier  d_mean", np.abs(mean - m32).max(), "d_std", np.abs(std - s32).max())
    assert np.abs(mean - m32).max() <= 1.5e-2
    assert np.abs(std - s32).max() <= 1.5e-2
    # the outputs are not degenerate (otherwise the comparison above would be vacuous)
    assert std[:, 1].min() > 1e-3 and 0.02 < mean[:, 1].min() and mean[:, 1].max() < 0.98


def test_philox_stream_equals_oracle_masks(iface, tiles):
    """counter-based Philox4x32-10 in the kernels == oracle.keep_masks: identical outputs bit for bit"""
    for base in (0, 5, (1 << 32) + 3):
        masks = X.keep_masks(N_TILES, T, 1024, 0.1, SEED, tile_index_base=base)
        a = iface.predict(tiles, T=T, masks=masks)
        b = iface.predict(tiles, T=T, seed=SEED, tile_index_base=base)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_reference_schedule_equivalence(weights, tiles):
    """the reference runs T FULL forward passes; one backbone pass + T head passes is identical"""
    o = X.XceptionUQOracle(weights, emulate_bf16=False)
    masks = X.keep_masks(2, 3, 1024, 0.1, 7)
    a = o.predict_uq(tiles[:2], T=3, masks=masks, reference_schedule=True)
    b = o.predict_uq(tiles[:2], T=3, masks=masks, reference_schedule=False)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_independent_masks_statistical_tolerance(iface, tiles):
    m1, s1 = iface.predict(tiles, T=100, seed=1)
    m2, s2 = iface.predict(tiles, T=100, seed=2)
    assert not np.array_equal(m1, m2)
    tol = 6.0 * np.maximum(s1, s2)[:, 1] / np.sqrt(100.0) + 1e-4
    assert (np.abs(m1[:, 1] - m2[:, 1]) <= tol).all(), (m1[:, 1], m2[:, 1], tol)
    assert np.abs(s1[:, 1] - s2[:, 1]).max() <= 0.5 * np.maximum(s1, s2)[:, 1].max()


def test_micro_batch_and_shard_invariance(weights, tiles, iface):
    """results do not depend on the micro-batch size nor on how tiles are sharded (tile_index_base)"""
    from biscuit_b200.uq import UncertaintyInterface
    big = UncertaintyInterface(weights, max_batch=8)
    a = iface.predict(tiles, T=T, seed=SEED)
    b = big.predict(tiles, T=T, seed=SEED)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    lo = big.predict(tiles[:2], T=T, seed=SEED, tile_index_base=0)
    hi = big.predict(tiles[2:], T=T, seed=SEED, tile_index_base=2)
    assert np.array_equal(np.concatenate([lo[0], hi[0]]), a[0])
    assert np.array_equal(np.concatenate([lo[1], hi[1]]), a[1])
    big.close()


def test_sample_sweep_and_call_surface(iface, tiles):
    for t in (1, 10, 30, 100):
        mean, std = iface.predict(tiles[:3], T=t, seed=3)
        assert np.isfinite(mean).all() and np.isfinite(std).all()
        if t == 1:
            assert (std == 0).all()
    logits, unc = iface(tiles[:2])                     # reference call surface (results.py:257)
    assert logits.shape == (2, 2) and unc.shape == (2, 2)          # per-class std: the reference reads uncertainty[0][0]


def test_device_resident_tiles(iface, tiles):
    import torch
    d = torch.from_numpy(tiles).cuda()
    a = iface.predict(d, T=T, seed=SEED)
    b = iface.predict(tiles, T=T, seed=SEED)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_simt_debug_path_agrees(tmp_path):
    """BQ_GEMM=simt (plain CUDA-core GEMM, debug only) vs the default tcgen05 path: same bf16 inputs, fp32
    accumulation in a different order"""
    code = (
        "import numpy as np, sys\n"
        "from oracle import synth, xception_uq as X\n"
        "from biscuit_b200.uq import UncertaintyInterface\n"
        "i = UncertaintyInterface(X.make_weights(seed=1), max_batch=2)\n"
        "m, s, f = i.predict(synth.tiles_u8(2, seed=0), T=10, seed=5, return_features=True)\n"
        "np.save(sys.argv[1], np.concatenate([m.ravel(), s.ravel(), f.ravel()]))\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = []
    for mode in ("simt", "tcgen05"):
        path = str(tmp_path / f"bq_{mode}.npy")
        env = dict(os.environ, BQ_GEMM=mode, PYTHONPATH=root)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, cwd=root, timeout=600)
        outs.append(np.load(path))
    a, b = outs
    print("simt vs tcgen05: max d (mean/std)", np.abs(a[:8] - b[:8]).max(), "features", np.abs(a[8:] - b[8:]).max())
    assert np.abs(a[:8] - b[:8]).max() <= 3e-3
    assert np.abs(a[8:] - b[8:]).max() <= 2e-2 * np.abs(a[8:]).max()


@pytest.mark.parametrize("t_samples", [7, 32, 70])
def test_fused_head_sample_chunks_vs_oracle(iface, tiles, oracle_bf16, t_samples):
    """T < 32, T == 32 and T > 32 (sample chunks merged with Chan's formula) against the oracle head"""
    o, _, _ = oracle_bf16
    masks = X.keep_masks(N_TILES, t_samples, 1024, 0.1, 77)
    mean, std = iface.predict(tiles, T=t_samples, masks=masks)
    m_ref, s_ref = o.predict_uq(tiles, T=t_samples, masks=masks)
    assert np.abs(mean - m_ref).max() <= 4e-3 and np.abs(std - s_ref).max() <= 4e-3
    a = iface.predict(tiles, T=t_samples, seed=77)
    assert np.array_equal(a[0], mean) and np.array_equal(a[1], std)      # Philox == injected masks


def test_repeatable_at_production_batch():
    """Same tiles, same seed, production micro-batch (256) and more tiles than one batch: every run must be
    BIT-identical (features, mean, std).  Guards the persistent kernels' smem pipelines: a parity-aliasing bug in the
    depthwise ring once changed a few rows of ~5 % of the tiles from run to run while every small-batch parity test
    passed."""
    import torch
    from biscuit_b200.uq import UncertaintyInterface
    from biscuit_b200.weights import random_init
    n = 700
    it = UncertaintyInterface(random_init(seed=1), max_batch=256)
    try:
        base = torch.from_numpy(synth.tiles_u8(50, seed=2)).cuda()
        t = base.repeat(n // 50, 1, 1, 1).contiguous()
        outs = [it.predict(t, T=6, seed=3, return_features=True) for _ in range(4)]
    finally:
        it.close()
    for o in outs[1:]:
        for a, b, name in zip(outs[0], o, ("mean", "std", "features")):
            bad = np.nonzero(np.abs(a - b).reshape(n, -1).max(1) > 0)[0]
            assert a.tobytes() == b.tobytes(), f"{name}: {len(bad)} tiles differ between runs, first {bad[:8]}"
    # the 50 distinct tiles repeat 14 times across different micro-batch positions / SMs: copies must agree exactly
    f = outs[0][2].reshape(n // 50, 50, -1)
    assert all(f[0].tobytes() == f[k].tobytes() for k in range(1, n // 50)), "copies of the same tile differ"


def test_results_do_not_depend_on_micro_batch():
    """A tile's features / mean / std are a function of (tile, global tile index, seed) only: bit-identical for
    micro-batches of 96 and 256 tiles (different GEMM M tiling, different SM assignment, partial last batch)."""
    import torch
    from biscuit_b200.uq import UncertaintyInterface
    from biscuit_b200.weights import random_init
    n = 330
    t = torch.from_numpy(synth.tiles_u8(66, seed=6)).cuda().repeat(5, 1, 1, 1).contiguous()
    outs = []
    for B in (96, 256):
        it = UncertaintyInterface(random_init(seed=1), max_batch=B)
        try:
            outs.append(it.predict(t, T=9, seed=8, return_features=True))
        finally:
            it.close()
    for a, b, name in zip(outs[0], outs[1], ("mean", "std", "features")):
        bad = np.nonzero(np.abs(a - b).reshape(n, -1).max(1) > 0)[0]
        assert a.tobytes() == b.tobytes(), f"{name}: {len(bad)} tiles depend on the micro-batch size, first {bad[:8]}"


# ----------------------------------------------------------------------------------------------------------------
# The configuration bench.py times (max_batch = biscuit_b200.uq.BENCH_MICRO_BATCH: CUDA-graph replay, batched fused
# head, full-size GEMM rings) tied to the oracle
# ----------------------------------------------------------------------------------------------------------------
from biscuit_b200.uq import BENCH_MICRO_BATCH as BENCH_BATCH  # noqa: E402


@pytest.fixture(scope="module")
def bench_iface(weights):
    from biscuit_b200.uq import UncertaintyInterface
    it = UncertaintyInterface(weights, max_batch=BENCH_BATCH)
    yield it
    it.close()


def test_bench_micro_batch_bit_identical_to_small_batch(weights, bench_iface, iface):
    """530 tiles at the bench micro-batch (one full graph-replayed micro-batch + a partial one, fused head launched on
    >= 592-tile... here 530-tile batches) and the same tiles at max_batch = 4 (the batch size the stage-wise oracle
    parity tests run at): bit-identical features / mean / std.  Transitively ties the bench configuration to the
    oracle."""
    import torch
    n = 530
    base = synth.tiles_u8(53, seed=9, n_slides=4)
    t = torch.from_numpy(base).cuda().repeat(10, 1, 1, 1).contiguous()
    big = bench_iface.predict(t, T=T, seed=21, return_features=True)
    small = iface.predict(t, T=T, seed=21, return_features=True)
    for a, b, name in zip(big, small, ("mean", "std", "features")):
        bad = np.nonzero(np.abs(a - b).reshape(n, -1).max(1) > 0)[0]
        assert a.tobytes() == b.tobytes(), f"{name}: {len(bad)} tiles differ between max_batch {BENCH_BATCH} and 4, first {bad[:8]}"
    # a second call replays the captured graph: still identical
    again = bench_iface.predict(t, T=T, seed=21, return_features=True)
    assert all(a.tobytes() == b.tobytes() for a, b in zip(big, again))


def test_oracle_parity_at_bench_micro_batch(weights, bench_iface, tiles):
    """The bench micro-batch: the six oracle tiles scattered over a run of one full micro-batch + 8 tiles (first /
    interior / last row of the full micro-batch, and the partial second micro-batch) against the bf16-emulated oracle
    directly, own Philox stream addressed by the GLOBAL tile index."""
    n = BENCH_BATCH + 8
    pos = [0, 63, 257, BENCH_BATCH - 1, BENCH_BATCH, n - 1]
    filler = synth.tiles_u8(16, seed=33, n_slides=2)
    allt = np.concatenate([filler] * (n // 16 + 1))[:n].copy()
    for k, p in enumerate(pos):
        allt[p] = tiles[k]
    mean, std, feats = bench_iface.predict(allt, T=T, seed=SEED, return_features=True)
    o = X.XceptionUQOracle(weights, emulate_bf16=True)
    for k, p in enumerate(pos):
        m_ref, s_ref, f_ref = o.predict_uq(tiles[k:k + 1], T=T, seed=SEED, tile_index_base=p, return_features=True)
        assert np.abs(feats[p] - f_ref[0]).max() <= 3e-2 * np.abs(f_ref).max(), (p, np.abs(feats[p] - f_ref[0]).max())
        assert np.abs(mean[p] - m_ref[0]).max() <= 4e-3, (p, mean[p], m_ref[0])
        assert np.abs(std[p] - s_ref[0]).max() <= 4e-3, (p, std[p], s_ref[0])


def test_config1_end_to_end_512_tiles_4_slides(weights, bench_iface):
    """BASELINE.json configs[0] / SURVEY.md 8d config 1: 512 synthetic tiles = 4 slides x 128 (per-slide colour
    bias), labels slides 0,1 -> 0 and 2,3 -> 1, T = 30 -> `predict_table` -> `threshold.apply(tile_uq = q50 of the
    tile uncertainty, slide_uq = q75 of the slide uncertainty, tile_pred = slide_pred = .5)`.
    Model: per-tile mean / std within 4e-3 of the CPU restatement (bf16-emulated tier, one backbone pass -- identical to
    the reference schedule of T full passes, test_reference_schedule_equivalence).  Thresholding: include / exclude
    decisions, slide table and metrics BIT-equal to the oracle's `apply` on the GPU's own tile table."""
    import pandas as pd
    from biscuit_b200 import threshold
    from biscuit_b200.uq import predict_table
    from oracle import threshold_oracle as O
    from helpers import assert_same_df, assert_same_results
    n, n_slides = 512, 4
    t = synth.tiles_u8(n, seed=0, n_slides=n_slides)
    slides = np.repeat([f"slide{j}" for j in range(n_slides)], n // n_slides)
    y_true = np.repeat([0, 0, 1, 1], n // n_slides).astype(np.int64)
    df = predict_table(bench_iface, t, slides, y_true, T=T, seed=SEED)
    assert list(df.columns) == ["slide", "y_true", "y_pred", "uncertainty"] and len(df) == n
    assert df["y_pred"].dtype == np.float32 and df["uncertainty"].dtype == np.float32
    # model half vs the CPU restatement
    o = X.XceptionUQOracle(weights, emulate_bf16=True)
    m_ref, s_ref = o.predict_uq(t, T=T, seed=SEED)
    d_mean = np.abs(df["y_pred"].to_numpy() - m_ref[:, 1]).max()
    d_std = np.abs(df["uncertainty"].to_numpy() - s_ref[:, 1]).max()
    print("config 1: d_mean", d_mean, "d_std", d_std)
    assert d_mean <= 4e-3 and d_std <= 4e-3
    # thresholding half, bit-exact on the GPU's own table
    tile_uq = np.float64(np.quantile(df["uncertainty"].to_numpy().astype(np.float64), 0.5))
    slide_unc = df.groupby("slide", sort=False)["uncertainty"].mean().to_numpy().astype(np.float64)
    slide_uq = np.float64(np.quantile(slide_unc, 0.75))
    for level, keep in (("slide", "high_confidence"), ("slide", "low_confidence")):
        kw = dict(tile_uq=tile_uq, slide_uq=slide_uq, tile_pred=0.5, slide_pred=0.5, keep=keep, level=level)
        a, b = df.copy(), df.copy()
        r_ref, s_ref_df = O.apply(a, **kw)
        r_gpu, s_gpu_df = threshold.apply(b, **kw)
        assert_same_results(r_ref, r_gpu, f"config1 {keep}")
        assert_same_df(s_ref_df, s_gpu_df, f"config1 {keep}")
        assert_same_df(a, b, f"config1 mutated tile table {keep}")
    # the decisions also agree with thresholding the ORACLE's predictions wherever no value sits within tolerance of a cut
    ref_tab = pd.DataFrame({"slide": slides, "y_true": y_true, "y_pred": m_ref[:, 1], "uncertainty": s_ref[:, 1]})
    r2, s2 = O.apply(ref_tab, tile_uq=tile_uq, slide_uq=slide_uq, tile_pred=0.5, slide_pred=0.5)
    r1, s1 = threshold.apply(df.copy(), tile_uq=tile_uq, slide_uq=slide_uq, tile_pred=0.5, slide_pred=0.5)
    if s1 is not None and s2 is not None:
        far = np.abs(s2["uncertainty"].to_numpy().astype(np.float64) - slide_uq) > 4e-3
        common = [s for s in s2["slide"][far] if s in set(s1["slide"])]
        assert len(common) == int(far.sum()), (list(s1["slide"]), list(s2["slide"]))


def test_fused_middle_flow_agrees_with_separate_kernels(tmp_path):
    """Default: the 728-wide middle flow runs in `sepconv_mid_kernel` (depthwise produced on-chip into the N-side
    operand of a transposed cta_group::2 GEMM, zero-padded flattened layout).  BQ_SEPMID=off: stand-alone depthwise
    kernel + pointwise GEMM.  Same bf16 rounding points and the same fp32 depthwise tap order; only the tensor-core
    accumulation order may differ -> bf16-level agreement on the features (and usually bit-identity)."""
    code = (
        "import numpy as np, sys, torch\n"
        "from oracle import synth\n"
        "from biscuit_b200.weights import random_init\n"
        "from biscuit_b200.uq import UncertaintyInterface\n"
        "i = UncertaintyInterface(random_init(seed=1), max_batch=48)\n"
        "t = torch.from_numpy(synth.tiles_u8(25, seed=4)).cuda().repeat(5, 1, 1, 1).contiguous()\n"
        "m, s, f = i.predict(t, T=5, seed=5, return_features=True)\n"
        "b12 = i.debug_stage(synth.tiles_u8(3, seed=4), 'block12')\n"
        "np.save(sys.argv[1], np.concatenate([m.ravel(), s.ravel(), f.ravel(), b12.ravel()]))\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = []
    for mode in ("off", "on"):
        path = str(tmp_path / f"bq_sepmid_{mode}.npy")
        env = dict(os.environ, BQ_SEPMID=mode, PYTHONPATH=root)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, cwd=root, timeout=600)
        outs.append(np.load(path))
    a, b = outs
    n = 125
    d = np.abs(a - b)
    print("sepmid on vs off: bit-identical" if a.tobytes() == b.tobytes() else
          f"sepmid on vs off: max d mean/std {d[:4 * n].max():.3e}, features {d[4 * n:4 * n + n * 2048].max():.3e}, block12 {d[4 * n + n * 2048:].max():.3e}")
    assert d[:4 * n].max() <= 3e-3
    f = a[4 * n:4 * n + n * 2048]
    assert d[4 * n:4 * n + n * 2048].max() <= 2e-2 * np.abs(f).max()
    b12 = a[4 * n + n * 2048:]
    assert d[4 * n + n * 2048:].max() <= 3e-2 * np.abs(b12).max()


@pytest.mark.parametrize("sites", [(True, True, True), (True, False, True), (False, False, True)])
def test_dropout_site_placements_vs_oracle(weights, tiles, oracle_bf16, sites):
    """MC-dropout placement is a model property that depends on the Slideflow version (SURVEY.md App. B):
    `ModelConfig.dropout_sites` = (after the pooled 2048-d features, after hidden_0, after hidden_1).  With site 0 on,
    hidden_0 is evaluated per (tile, sample) on the masked features.  Injected masks vs the oracle's head, and the
    kernels' own Philox stream == the oracle's masks, for every placement."""
    from biscuit_b200.hp import nature2022
    from biscuit_b200.uq import UncertaintyInterface
    cfg = nature2022.replace(dropout_sites=sites)
    it = UncertaintyInterface(weights, config=cfg, max_batch=4)
    try:
        enabled = [i for i, on in enumerate(sites) if on]
        width = 2048 if sites[0] else 1024
        masks = X.keep_masks(N_TILES, T, width, 0.1, SEED, sites=enabled)
        mean, std = it.predict(tiles, T=T, masks=masks)
        o = X.XceptionUQOracle(weights, emulate_bf16=True, dropout_sites=sites)
        m_ref, s_ref = o.predict_uq(tiles, T=T, masks=masks)
        print(sites, "d_mean", np.abs(mean - m_ref).max(), "d_std", np.abs(std - s_ref).max())
        assert np.abs(mean - m_ref).max() <= 4e-3 and np.abs(std - s_ref).max() <= 4e-3
        own = it.predict(tiles, T=T, seed=SEED)
        assert np.array_equal(own[0], mean) and np.array_equal(own[1], std)      # Philox stream == injected masks
        # a different placement gives a different answer (the option is not a no-op)
        base, _, _ = oracle_bf16
        m_def, s_def = base.predict_uq(tiles, T=T, seed=SEED)
        assert np.abs(s_ref - s_def).max() > 1e-4
        # sample counts beyond one 32-slot chunk, partial micro-batch
        m70 = X.keep_masks(N_TILES, 70, width, 0.1, 5, sites=enabled)
        a = it.predict(tiles, T=70, masks=m70)
        b = o.predict_uq(tiles, T=70, masks=m70)
        assert np.abs(a[0] - b[0]).max() <= 4e-3 and np.abs(a[1] - b[1]).max() <= 4e-3
    finally:
        it.close()


def test_dropout_sites_config_errors(weights):
    from biscuit_b200.hp import nature2022
    from biscuit_b200.uq import UncertaintyInterface
    with pytest.raises(ValueError):
        UncertaintyInterface(weights, config=nature2022.replace(dropout_sites=(True, True)), max_batch=2)
    it = UncertaintyInterface(weights, config=nature2022.replace(dropout_sites=(True, True, True)), max_batch=2)
    try:
        with pytest.raises(ValueError):                           # masks of the default placement's shape are rejected
            it.predict(np.zeros((1, 299, 299, 3), np.uint8), T=2, masks=np.ones((1, 2, 2, 1024), np.uint8))
    finally:
        it.close()


def test_standardized_float_input_is_the_reference_call(iface, tiles, oracle_bf16):
    """The reference's literal call site (results.py:249-258): `parsed = tf.image.per_image_standardization(tile)`,
    `logits, uncertainty = interface(tf.expand_dims(parsed, 0))`, `uncertainty[0][0]`.  A float32 batch standardised by
    the caller (here: the oracle's restatement of per_image_standardization) must give what the fused uint8 path gives, up
    to the fp32 rounding of computing (x - mean) * (1 / std) on the host instead of in the kernel."""
    o, _, _ = oracle_bf16
    parsed = o.standardize(tiles[:3]).permute(0, 2, 3, 1).contiguous().numpy()          # float32 NHWC, standardised
    assert parsed.dtype == np.float32 and abs(float(parsed[0].mean())) < 1e-3
    m_f, s_f, f_f = iface.predict(parsed, T=T, seed=SEED, return_features=True)
    m_u, s_u, f_u = iface.predict(tiles[:3], T=T, seed=SEED, return_features=True)
    assert np.abs(f_f - f_u).max() <= 2e-2 * np.abs(f_u).max()
    assert np.abs(m_f - m_u).max() <= 3e-3 and np.abs(s_f - s_u).max() <= 3e-3
    logits, uncertainty = iface(parsed[:1], T=T, seed=SEED)
    assert logits.shape == (1, 2) and float(uncertainty[0][0]) == float(s_f[0, 0])
    with pytest.raises(TypeError):
        iface.predict(tiles[:1].astype(np.int32))
    with pytest.raises(ValueError):
        iface.predict(tiles[:2], out_mean=np.empty((2, 2), np.float64))
