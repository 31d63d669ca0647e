"""CPU tier for the nested-CV caller (SURVEY.md 8f rank 1): pins oracle/nested_cv_oracle.py against the committed
outputs of the unmodified reference (tests/golden/nested_cv_golden.json) and, in the build container, against the live
reference; checks the host-side loaders / model lookup of biscuit_b200.utils (no GPU needed: pure pandas + os)."""
import importlib
import os
import warnings

import pandas as pd
import pytest

from oracle import nested_cv_oracle as NO, synth
from oracle.ref_shim import load_reference, reference_available

from helpers import load_golden
from nested_cv_common import assert_matches_golden, assert_same_outputs, build_case

warnings.simplefilter("ignore")
GOLD = load_golden("nested_cv_golden.json")


@pytest.mark.parametrize("name", sorted(GOLD["cases"]))
def test_oracle_matches_golden(name, tmp_path):
    case = GOLD["cases"][name]
    project, call = build_case(tmp_path, case["kwargs"])
    df, th = NO.thresholds_from_nested_cv(project, "EXP_AA_UQ", **call)
    assert_matches_golden(df, th, case, name)


@pytest.mark.skipif(not reference_available(), reason="needs a checkout of the original biscuit project in BISCUIT_REFERENCE_ROOT")
def test_live_reference_matches_oracle(tmp_path):
    load_reference()
    import slideflow as sf
    ref_exp = importlib.import_module("biscuit.experiment")
    plain = synth.nested_cv_project(str(tmp_path), seed0=1300, n_slides=30, tiles_per_slide=40)
    proj = type("P", (sf.Project, synth.FakeProject), {})(plain.models_dir, plain._patients)
    ref = ref_exp.Experiment(proj, outcome="cohort").thresholds_from_nested_cv("EXP_AA_UQ")
    mine = NO.thresholds_from_nested_cv(plain, "EXP_AA_UQ")
    assert_same_outputs(ref, mine, "live reference vs oracle")


def test_loaders_and_model_lookup(tmp_path):
    from biscuit_b200 import utils
    from biscuit_b200.errors import MatchError, ModelNotFoundError, MultipleModelsFoundError
    project = synth.nested_cv_project(str(tmp_path), outer_k=2, inner_k=3, n_slides=6, tiles_per_slide=5, seed0=40,
                                      fmt="parquet", underscore=True)
    assert issubclass(ModelNotFoundError, MatchError) and issubclass(MultipleModelsFoundError, MatchError)
    folder = utils.find_model(project, "EXP_AA_UQ", "cohort", kfold=2)
    assert os.path.basename(folder)[6:] == "cohort-EXP_AA_UQ-HP0-kfold2"
    assert utils.find_model(project, "EXP_AA_UQ", "cohort", kfold=2, epoch=1) == \
        os.path.join(folder, "cohort-EXP_AA_UQ-HP0-kfold2_epoch1")
    assert utils.model_exists(project, "EXP_AA_UQ-k1", "cohort", kfold=3)
    assert not utils.model_exists(project, "EXP_AA_UQ-k1", "cohort", kfold=4)
    with pytest.raises(ModelNotFoundError):
        utils.find_cv(project, "EXP_AA_UQ-k1", "cohort", k=4)
    os.makedirs(os.path.join(project.models_dir, "99999-cohort-EXP_AA_UQ-HP0-kfold2"))
    with pytest.raises(MultipleModelsFoundError):
        utils.find_model(project, "EXP_AA_UQ", "cohort", kfold=2)
    dfs = utils.df_from_cv(project, "EXP_AA_UQ-k1", "cohort", k=3)
    ref = NO.df_from_cv(project, "EXP_AA_UQ-k1", "cohort", 3)
    assert len(dfs) == 3
    for a, b in zip(dfs, ref):
        pd.testing.assert_frame_equal(a, b)
        assert {"y_true", "y_pred", "uncertainty", "slide", "patient"} <= set(a.columns)
        assert str(a["y_pred"].dtype) == "float32"          # parquet keeps the model's float32
    assert len(utils.slides_from_model_manifest(folder)) == 4 * 6
    assert len(utils.slides_from_model_manifest(folder, dataset="validation")) == 6
    assert len(utils.slides_from_model_manifest(os.path.join(folder, "cohort-EXP_AA_UQ-HP0-kfold2_epoch1"))) == 24
    with pytest.raises(OSError):
        utils.read_tile_predictions(os.path.join(folder, "predictions.txt"))
    with pytest.raises(ValueError):
        from biscuit_b200.experiment import Experiment
        Experiment("/some/path")
