"""CPU tier: pin the oracle (oracle/threshold_oracle.py) against
  (1) the committed outputs of the unmodified reference (tests/golden/threshold_golden.json),
  (2) the live reference through oracle/ref_shim.py when BISCUIT_REFERENCE_ROOT names a checkout of it,
  (3) the installed sklearn / pandas / numpy for the library-free tier the kernels implement.
"""
import warnings

import numpy as np
import pandas as pd
import pytest
from sklearn import metrics

from oracle import synth, threshold_oracle as O
from oracle.make_golden import CASES, make_table
from oracle.ref_shim import load_reference, reference_available

from helpers import assert_same_df, assert_same_results, dec, df_sha, load_golden, same_scalar

warnings.simplefilter("ignore")
GOLD = load_golden()


def test_versions_match_golden():
    import sklearn
    v = GOLD["versions"]
    assert (np.__version__, pd.__version__, sklearn.__version__) == (v["numpy"], v["pandas"], v["sklearn"]), \
        "golden vectors were generated with a different numpy/pandas/sklearn stack"


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_golden(name):
    case = GOLD["cases"][name]
    df = make_table(CASES[name])
    assert len(df) == case["n_rows"]
    th, auc = O.detect(df.copy())
    for k, v in case["detect"]["thresholds"].items():
        assert same_scalar(th[k], dec(v)), (name, k, th[k], dec(v))
    assert same_scalar(auc, dec(case["detect"]["auc"]))
    if th["tile_uq"] is None or th["slide_uq"] is None:
        th = {"tile_uq": 0.05, "slide_uq": 0.03, "tile_pred": 0.5, "slide_pred": 0.5}
    pats = synth.patients_map(df)
    for key, g in case["apply"].items():
        level, keep = key.split("/")
        d2 = df.copy()
        res, s_df = O.apply(d2, **th, keep=keep, patients=pats, level=level)
        assert_same_results(res, {k: dec(v) for k, v in g["results"].items()}, f"{name}/{key}")
        assert df_sha(s_df) == g["s_df"]["sha256"], f"{name}/{key}: group frame differs"
        assert df_sha(d2) == g["tile_df_sha256"], f"{name}/{key}: mutated tile frame differs"
        assert [str(t) for t in s_df.dtypes] == g["s_df"]["dtypes"]
    res, s_df = O.apply(df.copy(), 0.045, 0.031, tile_pred=0.5, slide_pred=0.45)
    assert_same_results(res, {k: dec(v) for k, v in case["apply_pyfloat"]["results"].items()}, name)
    assert df_sha(s_df) == case["apply_pyfloat"]["s_df"]["sha256"]


def test_oracle_from_cv_matches_golden():
    g = GOLD["from_cv"]
    dfs = synth.cv_tables(**g["kwargs"])
    r = O.from_cv([d.copy() for d in dfs])
    assert_same_results(r, {k: dec(v) for k, v in g["all_detect"].items()})
    r1 = O.from_cv([d.copy() for d in dfs], tile_uq="detect", slide_uq=None, tile_pred="detect",
                   slide_pred="detect")
    assert_same_results(r1, {k: dec(v) for k, v in g["tile_only"].items()})
    r2 = O.from_cv([d.copy() for d in dfs], tile_uq=r1["tile_uq"], slide_uq="detect", tile_pred="detect",
                   slide_pred="detect")
    assert_same_results(r2, {k: dec(v) for k, v in g["nested_second"].items()})


@pytest.mark.skipif(not reference_available(), reason="needs a checkout of the original biscuit project in BISCUIT_REFERENCE_ROOT")
def test_oracle_matches_live_reference():
    R = load_reference().threshold
    for seed in range(16):
        kw = dict(n_slides=10 + seed, tiles_per_slide=25 + 3 * seed, seed=seed,
                  dtype=[np.float32, np.float64][seed % 2], ties=[None, 40][seed % 3 == 0],
                  shuffle=seed % 4 == 1, ragged=seed % 5 == 2, slides_per_patient=1 + seed % 3)
        df = synth.tile_table(**kw)
        a, b = df.copy(), df.copy()
        ra, rb = R.detect(a), O.detect(b)
        assert_same_results(ra[0], rb[0], f"detect seed {seed}")
        assert same_scalar(ra[1], rb[1])
        assert_same_df(a, b, f"detect-mutated seed {seed}")
        th = ra[0]
        if th["tile_uq"] is None or th["slide_uq"] is None:
            th = dict(tile_uq=0.05, slide_uq=0.03, tile_pred=0.5, slide_pred=0.5)
        pats = synth.patients_map(df)
        for level in ("slide", "patient"):
            for keep in ("high_confidence", "low_confidence"):
                a, b = df.copy(), df.copy()
                x = R.apply(a, **th, keep=keep, patients=pats, level=level)
                y = O.apply(b, **th, keep=keep, patients=pats, level=level)
                assert_same_results(x[0], y[0], f"apply seed {seed}")
                assert_same_df(x[1], y[1], f"apply s_df seed {seed}")
                assert_same_df(a, b, f"apply tile df seed {seed}")


@pytest.mark.skipif(not reference_available(), reason="needs a checkout of the original biscuit project in BISCUIT_REFERENCE_ROOT")
def test_reference_error_behaviour_matches_oracle():
    R = load_reference()
    df = synth.tile_table(8, 20, seed=3)
    bad = df.copy()
    bad.loc[3, "y_pred"] = np.nan
    with pytest.raises(R.errors.PredsContainNaNError):
        R.threshold.apply(bad.copy(), 0.05, 0.03)
    with pytest.raises(O.PredsContainNaNError):
        O.apply(bad.copy(), 0.05, 0.03)
    assert R.threshold.detect(bad.copy()) == O.detect(bad.copy()) == (
        {k: None for k in ("tile_uq", "slide_uq", "tile_pred", "slide_pred")}, None)
    with pytest.raises(TypeError):
        R.threshold.apply(df.copy(), None, 0.03)
    with pytest.raises(TypeError):
        O.apply(df.copy(), None, 0.03)
    # everything filtered out -> ({None...}, None)
    assert R.threshold.apply(df.copy(), 1e-9, 0.03)[1] is None
    assert O.apply(df.copy(), 1e-9, 0.03)[1] is None
    # perfectly separable tiles: the tile-UQ ROC is single-class -> the reference's Youden idiom
    # raises an uncaught ValueError (SURVEY App. A.1)
    sep = df.copy()
    sep["y_pred"] = sep["y_true"].astype(np.float32) * 0.8 + 0.1
    with pytest.raises(ValueError):
        R.threshold.from_cv([sep.copy()])
    with pytest.raises(ValueError):
        O.from_cv([sep.copy()])
    # some wrong tiles but every slide right -> slide_uq None -> fold skipped -> ThresholdError
    easy = df.copy()
    rng = np.random.default_rng(5)
    easy["y_pred"] = (0.5 + 0.1 * (2 * easy["y_true"] - 1) + rng.normal(0, 0.12, len(easy))).astype(np.float32)
    with pytest.raises(R.errors.ThresholdError):
        R.threshold.from_cv([easy.copy()])
    with pytest.raises(O.ThresholdError):
        O.from_cv([easy.copy()])


# --- tier 2: the library-free restatement the CUDA kernels follow ----------------------------------

def test_tier2_roc_youden_auc_match_sklearn():
    rng = np.random.default_rng(1)
    for trial in range(300):
        n = int(rng.integers(2, 300))
        dt = [np.float32, np.float64][trial % 2]
        s = rng.random(n).astype(dt)
        if trial % 3 == 0:
            s = (np.round(s * rng.integers(2, 20)) / 10).astype(dt)
        y = rng.integers(0, 2, n)
        if trial % 50 == 7:
            y[:] = 1
        if trial % 50 == 9:
            y[:] = 0
        fpr, tpr, thr = metrics.roc_curve(y, s)
        fps, tps, th2 = O.roc_points(y, s)
        f2, t2 = O.rates(fps, tps)
        assert np.array_equal(fpr, f2, equal_nan=True) and np.array_equal(tpr, t2, equal_nan=True)
        assert np.array_equal(thr, th2)
        try:
            a = O._youden_pick(fpr, tpr, thr)
        except ValueError:
            a = "VE"
        try:
            b = O.youden(fps, tps, th2)[0]
        except ValueError:
            b = "VE"
        assert a == b
        au, a2 = metrics.auc(fpr, tpr), O.trapezoid_auc(fps, tps)
        assert au == a2 or (au != au and a2 != a2)


def test_tier2_pairwise_sum_matches_numpy():
    rng = np.random.default_rng(2)
    for n in list(range(1, 40)) + [127, 128, 129, 130, 255, 256, 257, 1000, 1001, 4097]:
        a = rng.random(n) * rng.choice([1, 1e-3, 1e3], n)
        assert O.pairwise_sum(a) == np.sum(a)


def test_tier2_kahan_matches_pandas_group_mean():
    rng = np.random.default_rng(3)
    for trial in range(60):
        n, L = int(rng.integers(1, 2500)), int(rng.integers(1, 20))
        dt = [np.float32, np.float64][trial % 2]
        v = (rng.random(n) * rng.choice([1, 1e-4, 1e4], n)).astype(dt)
        g = rng.integers(0, L, n)
        ref = pd.DataFrame({"g": g, "v": v}).groupby("g").mean()["v"]
        out, _ = O.kahan_group_mean(v, g, L)
        for k in ref.index:
            assert ref[k] == out[k]
