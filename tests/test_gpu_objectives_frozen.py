"""Every objective against frozen outputs of the CUDA path (tests/golden/objective_outputs.json, written by
tests/golden/make_objective_outputs.py on a B200).  Exact equality of the model string, the training
metrics, the training scores (sha256 of their float64 bytes) and the constant-hessian flag: the oracle
tests allow 1e-5, which is too loose to show that a change to the objective code moved nothing."""
import importlib.util
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _maker():
    spec = importlib.util.spec_from_file_location("make_objective_outputs", os.path.join(GOLDEN, "make_objective_outputs.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


MAKER = _maker()
with open(os.path.join(GOLDEN, "objective_outputs.json")) as _f:
    FROZEN = json.load(_f)["cases"]


def test_every_case_is_frozen():
    assert sorted(FROZEN) == sorted(MAKER.CASES)


@pytest.mark.parametrize("name", sorted(MAKER.CASES))
def test_objective_outputs_unchanged(built, name):
    got = MAKER.run_case(name)
    want = FROZEN[name]
    assert got["model"] == want["model"]
    assert got["eval"] == want["eval"]
    assert got["scores_sha256"] == want["scores_sha256"]
    assert got["constant_hessian"] == want["constant_hessian"]


@pytest.mark.parametrize("objective", ["multiclass", "multiclassova"])
def test_reset_num_class_keeps_class_count(built, objective):
    """The class count is fixed when the booster is created: LGBM_BoosterResetParameter("num_class=...") between iterations
    must train exactly as without it (the scores and gradients are sized for the original count)."""
    from mmlspark_b200 import capi
    X, s, _ = MAKER.data()
    y = np.clip(np.floor(s + 1.5), 0, 2).astype(np.float32)
    params = "objective=%s num_class=3 %s" % (objective, MAKER.BASE)
    runs = []
    for reset in (False, True):
        ds = capi.Dataset.from_mat(X, MAKER.DS_PARAMS)
        ds.set_field("label", y)
        bst = capi.Booster(ds, params)
        for it in range(4):
            if reset and it == 2:
                bst.reset_parameter("num_class=2")
            bst.update_one_iter()
        runs.append((bst.save_model_to_string().split("\nparameters:\n")[0], bst.get_scores(0).tobytes(), bst.get_eval(0).tolist()))
        bst.free()
        ds.free()
    assert runs[0] == runs[1]
