"""Frozen outputs of the CUDA path for every objective: writes tests/golden/objective_outputs.json.

Each case trains a small seeded booster through the C ABI and records the model string, the training
metrics, the sha256 of the training scores and whether the booster reports a constant hessian.  The
values pin "unchanged", not "correct" (correctness is the oracle tests' job): any change to the
objective code that moves a single bit shows up here.  Needs a CUDA device and the built library.
Re-run on a B200, after build(): python tests/golden/make_objective_outputs.py"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "objective_outputs.json")
DS_PARAMS = "max_bin=255 is_pre_partition=True bin_construct_sample_cnt=200000 num_threads=0"
BASE = "num_leaves=7 learning_rate=0.1 min_data_in_leaf=20 verbosity=-1"
ITERS = 5
N, F = 4000, 12


def data():
    rng = np.random.default_rng(2024)
    X = rng.standard_normal((N, F))
    X[:, 2] = np.round(X[:, 2], 1)
    X[:, 3] = np.where(rng.random(N) < 0.1, np.nan, X[:, 3])
    s = X[:, 0] + 0.7 * np.nan_to_num(X[:, 3]) - 0.5 * X[:, 4] + X[:, 5] * X[:, 6] + 0.3 * rng.standard_normal(N)
    w = rng.uniform(0.2, 2.0, N)
    return X, s, w


def labels(kind, s):
    if kind == "real":
        return s
    if kind == "positive":
        return np.exp(0.5 * s)
    if kind == "binary":
        return (s > 0.5).astype(np.float64)
    if kind == "negatives":
        return np.zeros_like(s)
    if kind == "multiclass_gap":       # 4 classes, class 2 absent
        return np.array([0.0, 1.0, 3.0])[np.clip(np.floor(s + 1.5), 0, 2).astype(int)]
    if kind == "multiclass":
        return np.clip(np.floor(s + 2.0), 0, 3)
    if kind == "probability":
        return 1.0 / (1.0 + np.exp(-s))
    if kind == "relevance":
        return np.clip(np.floor(s + 2.0), 0, 4)
    raise ValueError(kind)


# name -> (params, label kind, options); options: weight, group, init_score, custom (one custom-gradient iteration first),
# reset (ResetParameter string applied after two iterations)
CASES = {
    "regression": ("objective=regression", "real", {}),
    "regression_weighted": ("objective=regression", "real", {"weight": True}),
    "regression_goss": ("objective=regression boosting_type=goss", "real", {}),
    "huber": ("objective=huber alpha=0.8", "real", {}),
    "fair": ("objective=fair fair_c=0.7", "real", {}),
    "poisson": ("objective=poisson", "positive", {}),
    "gamma": ("objective=gamma", "positive", {}),
    "tweedie": ("objective=tweedie tweedie_variance_power=1.3", "positive", {}),
    "regression_l1": ("objective=regression_l1", "real", {}),
    "quantile": ("objective=quantile alpha=0.7", "real", {}),
    "quantile_weighted": ("objective=quantile alpha=0.3", "real", {"weight": True}),
    "mape": ("objective=mape", "positive", {}),
    "binary_unbalance_spw": ("objective=binary is_unbalance=true scale_pos_weight=1.5", "binary", {}),
    "binary_all_negative": ("objective=binary", "negatives", {}),
    "multiclass_absent_class": ("objective=multiclass num_class=4", "multiclass_gap", {}),
    "multiclassova_unbalance": ("objective=multiclassova num_class=4 is_unbalance=true", "multiclass", {}),
    "cross_entropy_weighted": ("objective=cross_entropy", "probability", {"weight": True}),
    "lambdarank": ("objective=lambdarank lambdarank_truncation_level=5 lambdarank_norm=false", "relevance", {"group": True}),
    "regression_custom_first": ("objective=regression", "real", {"custom": True}),
    "binary_rf": ("objective=binary boosting_type=rf bagging_fraction=0.7 bagging_freq=1", "binary", {}),
    "regression_init_score": ("objective=regression", "real", {"init_score": True}),
    "huber_reset_alpha": ("objective=huber alpha=0.9", "real", {"reset": "alpha=0.5"}),
    "quantile_reset_alpha": ("objective=quantile alpha=0.6", "real", {"reset": "alpha=0.2"}),
}


def run_case(name):
    """Trains case `name` on the CUDA path and returns its record (JSON-ready)."""
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from mmlspark_b200 import capi
    params, kind, opt = CASES[name]
    X, s, w = data()
    y = labels(kind, s).astype(np.float32)
    ds = capi.Dataset.from_mat(X, DS_PARAMS)
    ds.set_field("label", y)
    if opt.get("weight"):
        ds.set_field("weight", w.astype(np.float32))
    if opt.get("group"):
        ds.set_field("group", np.full(N // 40, 40, dtype=np.int32))
    if opt.get("init_score"):
        ds.set_field("init_score", 0.1 * X[:, 7])
    bst = capi.Booster(ds, params + " " + BASE)
    done = 0
    if opt.get("custom"):
        g = (0.0 - y).astype(np.float32)       # L2 gradient at a zero score
        bst.update_one_iter_custom(g, np.ones(N, dtype=np.float32))
        done = ITERS - 2
    for it in range(done, ITERS):
        if opt.get("reset") and it == 2:
            bst.reset_parameter(opt["reset"])
        if bst.update_one_iter():
            break
    scores = np.ascontiguousarray(bst.get_scores(0), dtype=np.float64)
    rec = {"model": bst.save_model_to_string(),
           "eval": [float(v).hex() for v in bst.get_eval(0)],
           "scores_sha256": hashlib.sha256(scores.tobytes()).hexdigest(),
           "constant_hessian": bool(bst.get_info()["constant_hessian"])}
    bst.free()
    ds.free()
    return rec


def _first_line(cmd):
    try:
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True).stdout.strip().splitlines()
    except OSError:
        return ""
    return out[0] if out else ""


def main():
    # PRODUCER_COMMIT names the source commit when the tree is not a git checkout
    commit = os.environ.get("PRODUCER_COMMIT") or _first_line(["git", "rev-parse", "HEAD"]) or "unknown"
    gpu = _first_line(["nvidia-smi", "--query-gpu=name", "--format=csv,noheader"]) or "unknown"
    out = {"producer": {"commit": commit, "gpu": gpu},
           "cases": {name: run_case(name) for name in CASES}}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote %s (%d cases)" % (OUT, len(CASES)))


if __name__ == "__main__":
    main()
