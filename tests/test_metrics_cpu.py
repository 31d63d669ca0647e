"""CPU tier for the evaluation metrics (SURVEY.md 8f rank 4): pins oracle/metrics_oracle.py against the committed outputs of the
unmodified reference (tests/golden/metrics_golden.json) and, in the build container, against the live reference
(`np.float` alias restored for the call -- the reference's delong.py predates NumPy 1.24)."""
import warnings

import numpy as np
import pytest

from oracle import metrics_oracle as MO
from oracle.ref_shim import load_reference, reference_available

from helpers import dec, load_golden, same_scalar

warnings.simplefilter("ignore")
GOLD = load_golden("metrics_golden.json")


def check(res, dl, case, what):
    for k, v in case["metrics"].items():
        got = res[k]
        assert same_scalar(None if got is None else np.float64(got), dec(v)), (what, k, got, dec(v))
    if case["delong"] is not None:
        assert same_scalar(np.float64(dl[0]), dec(case["delong"][0])), (what, "auc", dl[0])
        assert same_scalar(np.float64(dl[1]), dec(case["delong"][1])), (what, "var", dl[1])


@pytest.mark.parametrize("name", sorted(MO.CASES))
def test_oracle_matches_golden(name):
    kw = MO.CASES[name]
    y, p, thr = MO.make_case(kw)
    np.random.seed(kw["seed"])
    res = MO.prediction_metrics(y, p, thr)
    dl = None if kw.get("single") else MO.delong_roc_variance(y, p)
    check(res, dl, GOLD["cases"][name], name)


@pytest.mark.skipif(not reference_available(), reason="needs a checkout of the original biscuit project in BISCUIT_REFERENCE_ROOT")
def test_live_reference_matches_oracle():
    R = load_reference()
    rng = np.random.default_rng(77)
    y = rng.integers(0, 2, 333).astype(np.int64)
    p = np.round(np.clip(0.5 + 0.2 * (2 * y - 1) + rng.normal(0, 0.3, 333), 0, 1) * 64) / 64
    for dtype in (np.float32, np.float64):
        np.random.seed(5)
        with MO.reference_with_np_float():
            ref = R.utils.prediction_metrics(y, p.astype(dtype), 0.5)
            ref_dl = R.delong.delong_roc_variance(y, p.astype(dtype))
        np.random.seed(5)
        mine = MO.prediction_metrics(y, p.astype(dtype), 0.5)
        mine_dl = MO.delong_roc_variance(y, p.astype(dtype))
        for k in ref:
            assert same_scalar(np.float64(ref[k]), np.float64(mine[k])), (k, ref[k], mine[k])
        assert float(ref_dl[0]) == float(mine_dl[0]) and float(ref_dl[1]) == float(mine_dl[1])


@pytest.mark.parametrize("name", sorted(MO.DELONG_TEST_CASES))
def test_delong_test_oracle_matches_golden(name):
    """two-classifier DeLong test (reference delong.py:110-123): the oracle restatement vs the reference's committed output"""
    g = load_golden("delong_test_golden.json")["cases"][name]
    y, a, b = MO.make_delong_test_case(MO.DELONG_TEST_CASES[name])
    lp = MO.delong_roc_test(y, a, b)
    assert list(lp.shape) == g["shape"] and same_scalar(np.float64(lp[0, 0]), dec(g["log10_p"])), (lp, dec(g["log10_p"]))
