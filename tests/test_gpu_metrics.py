"""Device-side evaluation (LGBM_BoosterGetEval; TrainUtils.scala:125-151 drives early stopping with it) against independent numpy /
scikit-learn restatements of the LightGBM metric definitions, on the training scores (data_idx 0) and a validation set (data_idx 1)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DS_PARAMS = "max_bin=255 is_pre_partition=True bin_construct_sample_cnt=200000 num_threads=0"
BASE = "num_leaves=15 learning_rate=0.2 min_data_in_leaf=20 verbosity=-1 "


def _fit(X, y, params, Xv=None, yv=None, weight=None, wv=None, group=None, gv=None, iters=5):
    from mmlspark_b200 import capi
    ds = capi.Dataset.from_mat(X, DS_PARAMS).set_field("label", y)
    if weight is not None:
        ds.set_field("weight", weight)
    if group is not None:
        ds.set_field("group", group)
    b = capi.Booster(ds, BASE + params)
    dv = None
    if Xv is not None:
        dv = capi.Dataset.from_mat(Xv, DS_PARAMS, reference=ds).set_field("label", yv)
        if wv is not None:
            dv.set_field("weight", wv)
        if gv is not None:
            dv.set_field("group", gv)
        b.add_valid(dv)
    for _ in range(iters):
        b.update_one_iter()
    return b, ds, dv


def _wavg(loss, w):
    w = np.ones_like(loss) if w is None else w.astype(np.float64)
    return float((loss * w).sum() / w.sum())


def test_binary_metrics_incl_weighted_auc_with_ties(built):
    from sklearn.metrics import roc_auc_score
    rng = np.random.default_rng(1)
    n = 30000
    X = np.round(rng.standard_normal((n, 6)), 1)            # coarse features => many tied scores
    y = (X[:, 0] + 0.5 * X[:, 1] + 0.8 * rng.standard_normal(n) > 0).astype(np.float32)
    w = (0.5 + rng.random(n)).astype(np.float32)
    Xv, yv, wv = X[:7000] + 0.1, y[:7000], w[:7000]
    b, _, _ = _fit(X, y, "objective=binary metric=auc,binary_logloss,binary_error", Xv, yv, w, wv, iters=3)
    assert b.eval_names() == ["auc", "binary_logloss", "binary_error"]
    for idx, (yy, ww) in enumerate(((y, w), (yv, wv))):
        s = b.get_scores(idx)
        p = 1.0 / (1.0 + np.exp(-s))
        got = b.get_eval(idx)
        assert len(np.unique(s)) < len(s) / 4                # the tie groups really occur
        np.testing.assert_allclose(got[0], roc_auc_score(yy, s, sample_weight=ww), rtol=1e-10)
        pl = np.where(yy > 0, p, 1 - p)
        np.testing.assert_allclose(got[1], _wavg(-np.log(np.maximum(pl, 1e-15)), ww), rtol=1e-12)
        np.testing.assert_allclose(got[2], _wavg(((p <= 0.5) == (yy > 0)).astype(np.float64), ww), rtol=1e-12)


def test_regression_metrics(built):
    rng = np.random.default_rng(2)
    n = 20000
    X = rng.standard_normal((n, 5))
    y = (np.exp(0.3 * X[:, 0]) + 0.1 * np.abs(rng.standard_normal(n))).astype(np.float32)
    w = (0.5 + rng.random(n)).astype(np.float32)
    names = "l2,rmse,l1,huber,fair,quantile,mape,poisson,tweedie"
    b, _, _ = _fit(X, y, "objective=regression alpha=0.7 fair_c=1.3 tweedie_variance_power=1.4 metric=" + names, weight=w)
    s = b.get_scores(0)
    got = dict(zip(b.eval_names(), b.get_eval(0)))
    d = s - y
    want = {
        "l2": _wavg(d * d, w), "rmse": np.sqrt(_wavg(d * d, w)), "l1": _wavg(np.abs(d), w),
        "huber": _wavg(np.where(np.abs(d) <= 0.7, 0.5 * d * d, 0.7 * (np.abs(d) - 0.35)), w),
        "fair": _wavg(1.3 * np.abs(d) - 1.69 * np.log(1 + np.abs(d) / 1.3), w),
        "quantile": _wavg(np.where(y - s < 0, (0.7 - 1) * (y - s), 0.7 * (y - s)), w),
        "mape": _wavg(np.abs(y - s) / np.maximum(1.0, np.abs(y)), w),
        "poisson": _wavg(np.maximum(np.exp(s), 1e-10) - y * np.log(np.maximum(np.exp(s), 1e-10)), w),
        "tweedie": _wavg(-y * np.exp((1 - 1.4) * np.log(np.maximum(np.exp(s), 1e-10))) / (1 - 1.4) + np.exp((2 - 1.4) * np.log(np.maximum(np.exp(s), 1e-10))) / (2 - 1.4), w),
    }
    for k, v in want.items():
        np.testing.assert_allclose(got[k], v, rtol=1e-11, err_msg=k)


@pytest.mark.parametrize("objective", ["multiclass", "multiclassova"])
def test_multiclass_metrics(built, objective):
    rng = np.random.default_rng(3)
    n, K = 20000, 4
    X = rng.standard_normal((n, 6))
    y = np.argmax(X[:, :K] + 0.7 * rng.standard_normal((n, K)), axis=1).astype(np.float32)
    b, _, _ = _fit(X, y, "objective=%s num_class=4 metric=multi_logloss,multi_error" % objective)
    s = b.get_scores(0).reshape(K, n).T
    if objective == "multiclass":
        e = np.exp(s - s.max(axis=1, keepdims=True))
        p = e / e.sum(axis=1, keepdims=True)
    else:
        p = 1.0 / (1.0 + np.exp(-s))
    pl = p[np.arange(n), y.astype(int)]
    got = b.get_eval(0)
    np.testing.assert_allclose(got[0], np.mean(-np.log(np.maximum(pl, 1e-15))), rtol=1e-12)
    np.testing.assert_allclose(got[1], np.mean((p >= pl[:, None]).sum(axis=1) > 1), rtol=1e-12)


def _rank_metrics(s, y, sizes, ks, gain):
    nd, mp = np.zeros(len(ks)), np.zeros(len(ks))
    off = 0
    for c in sizes:
        ss, yy = s[off:off + c], y[off:off + c].astype(int)
        off += c
        order = np.argsort(-ss, kind="stable")
        ideal = np.sort(yy)[::-1]
        npos = int((yy > 0.5).sum())
        for e, k in enumerate(ks):
            kk = min(k, c)
            disc = 1.0 / np.log2(2.0 + np.arange(kk))
            maxdcg = float((gain[ideal[:kk]] * disc).sum())
            nd[e] += 1.0 if maxdcg <= 0 else float((gain[yy[order[:kk]]] * disc).sum()) / maxdcg
            hits = (yy[order[:kk]] > 0.5)
            ap = float((np.cumsum(hits)[hits] / (np.nonzero(hits)[0] + 1.0)).sum())
            mp[e] += ap / min(npos, kk) if npos > 0 else 1.0
    return nd / len(sizes), mp / len(sizes)


def test_ranking_metrics_ndcg_and_map(built):
    rng = np.random.default_rng(4)
    sizes = rng.integers(1, 60, 800).astype(np.int32)
    sizes[5] = 300                                          # one query longer than the block
    n = int(sizes.sum())
    X = np.round(rng.standard_normal((n, 5)), 1)
    y = np.clip(np.round(X[:, 0] + 0.7 * rng.standard_normal(n) + 1.0), 0, 4).astype(np.float32)
    y[:sizes[0]] = 0                                        # an all-irrelevant query: ndcg = map = 1 by definition
    ks = [1, 3, 5, 10]
    # validation set = a prefix made of whole queries
    cut = int(np.searchsorted(np.cumsum(sizes), n // 2, side="right"))
    from mmlspark_b200 import capi
    nv = int(sizes[:cut].sum())
    ds = capi.Dataset.from_mat(X, DS_PARAMS).set_field("label", y).set_field("group", sizes)
    dv = capi.Dataset.from_mat(X[:nv], DS_PARAMS, reference=ds).set_field("label", y[:nv]).set_field("group", sizes[:cut])
    b = capi.Booster(ds, BASE + "objective=lambdarank metric=ndcg,map eval_at=1,3,5,10 min_data_in_leaf=5")
    b.add_valid(dv)
    for _ in range(4):
        b.update_one_iter()
    assert b.eval_names() == ["ndcg@1", "ndcg@3", "ndcg@5", "ndcg@10", "map@1", "map@3", "map@5", "map@10"]
    gain = np.array([0.0] + [float((1 << i) - 1) for i in range(1, 31)])
    for idx, (nn, sz) in enumerate(((n, sizes), (nv, sizes[:cut]))):
        s = b.get_scores(idx)
        nd, mp = _rank_metrics(s, y[:nn], sz, ks, gain)
        got = b.get_eval(idx)
        np.testing.assert_allclose(got[:4], nd, rtol=1e-10)
        np.testing.assert_allclose(got[4:], mp, rtol=1e-6)          # [UPSTREAM] accumulates num_hit / (j + 1.0f) in float


def _rank_case(rng, max_label):
    """single-document queries, short ones and one 1000-document query full of tied scores; a validation set of whole queries"""
    sizes = np.concatenate([np.ones(40, dtype=np.int32), rng.integers(2, 60, 300).astype(np.int32), [1000]]).astype(np.int32)
    rng.shuffle(sizes)
    n = int(sizes.sum())
    X = np.round(rng.standard_normal((n, 5)), 1)
    y = np.clip(np.round((X[:, 0] + 0.7 * rng.standard_normal(n) + 1.0) * max_label / 4), 0, max_label).astype(np.float32)
    cut = int(np.searchsorted(np.cumsum(sizes), n // 2, side="right"))
    return X, y, sizes, cut


EVAL_AT_16 = [1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 15, 20, 30, 50, 100, 2000]      # 2000: more than any query holds


@pytest.mark.parametrize("num_gain", [31, 40, 100])
def test_ranking_metrics_long_label_gain(built, num_gain):
    """k_metric_rank sizes its label histogram from label_gain: with 40 and 100 gains the labels above 63 count towards the max DCG"""
    rng = np.random.default_rng(num_gain)
    X, y, sizes, cut = _rank_case(rng, num_gain - 1)
    gain = _rank_gain(num_gain)
    nv = int(sizes[:cut].sum())
    lg = "" if num_gain == 31 else " label_gain=" + ",".join(repr(float(v)) for v in gain)
    params = "objective=lambdarank metric=ndcg,map eval_at=%s min_data_in_leaf=5%s" % (",".join(map(str, EVAL_AT_16)), lg)
    b, _, _ = _fit(X, y, params, X[:nv], y[:nv], group=sizes, gv=sizes[:cut], iters=3)
    assert b.eval_names() == ["ndcg@%d" % k for k in EVAL_AT_16] + ["map@%d" % k for k in EVAL_AT_16]
    assert y.max() == num_gain - 1
    for idx, (nn, sz) in enumerate(((len(y), sizes), (nv, sizes[:cut]))):
        s = b.get_scores(idx)
        nd, mp = _rank_metrics(s, y[:nn], sz, EVAL_AT_16, gain)
        got = b.get_eval(idx)
        np.testing.assert_allclose(got[:16], nd, rtol=1e-10)
        np.testing.assert_allclose(got[16:], mp, rtol=1e-6)


def _rank_gain(num_gain):
    if num_gain == 31:
        return np.array([0.0] + [float((1 << i) - 1) for i in range(1, 31)])
    return np.round(np.arange(num_gain, dtype=np.float64) ** 1.7, 4)


def test_map_negative_labels_are_not_relevant(built):
    """MAP counts label > 0.5 as relevant: -1 is not"""
    rng = np.random.default_rng(14)
    sizes = rng.integers(1, 40, 400).astype(np.int32)
    n = int(sizes.sum())
    X = np.round(rng.standard_normal((n, 5)), 1)
    y = rng.choice(np.array([-1, 0, 1, 2], dtype=np.float32), n, p=[0.4, 0.3, 0.2, 0.1])
    b, _, _ = _fit(X, y, "objective=regression metric=map eval_at=1,3,10,50", group=sizes, iters=2)
    nd, mp = _rank_metrics(b.get_scores(0), y, sizes, [1, 3, 10, 50], np.zeros(3))
    np.testing.assert_allclose(b.get_eval(0), mp, rtol=1e-6)


def test_ndcg_label_checks(built):
    """[LightGBM DCGCalculator::CheckLabel] on every dataset the ndcg metric evaluates: labels are integers in [0, label_gain.size())"""
    from mmlspark_b200 import capi
    rng = np.random.default_rng(15)
    n = 2000
    X = rng.standard_normal((n, 4))
    group = np.full(n // 20, 20, dtype=np.int32)
    y = rng.integers(0, 5, n).astype(np.float32)

    def train_set(labels):
        return capi.Dataset.from_mat(X, DS_PARAMS).set_field("label", labels).set_field("group", group)

    frac = y.copy()
    frac[17] = 1.5
    with pytest.raises(capi.LightGBMError, match="label should be int type"):
        capi.Booster(train_set(frac), BASE + "objective=regression metric=ndcg")
    with pytest.raises(capi.LightGBMError, match="label should be int type"):
        capi.Booster(train_set(frac), BASE + "objective=lambdarank")
    neg = y.copy()
    neg[3] = -1
    with pytest.raises(capi.LightGBMError, match="Label should be non-negative"):
        capi.Booster(train_set(neg), BASE + "objective=regression metric=ndcg")
    big = y.copy()
    big[9] = 40
    with pytest.raises(capi.LightGBMError, match=r"Label 40 is not less than the number of label mappings \(31\)"):
        capi.Booster(train_set(big), BASE + "objective=regression metric=ndcg")
    # a validation set whose labels fall outside label_gain is refused when it is added
    ds = train_set(y)
    b = capi.Booster(ds, BASE + "objective=lambdarank metric=ndcg label_gain=0,1,3,7,15")
    dv = capi.Dataset.from_mat(X, DS_PARAMS, reference=ds).set_field("label", np.where(np.arange(n) == 5, 5, y).astype(np.float32))
    dv.set_field("group", group)
    with pytest.raises(capi.LightGBMError, match=r"Label 5 is not less than the number of label mappings \(5\)"):
        b.add_valid(dv)
    # ... and so is a reset that shortens label_gain below the labels of a dataset already added
    b2 = capi.Booster(train_set(y), BASE + "objective=regression metric=l2")
    with pytest.raises(capi.LightGBMError, match=r"Label [34] is not less than the number of label mappings \(3\)"):
        b2.reset_parameter("metric=ndcg label_gain=0,1,3")
    assert b2.eval_names() == ["l2"] and len(b2.get_eval(0)) == 1              # the refused reset left the booster as it was
    # map alone does not index label_gain: negative and large labels are fine
    capi.Booster(train_set(np.where(np.arange(n) % 7 == 0, -1, 70).astype(np.float32)), BASE + "objective=regression metric=map").get_eval(0)


def test_unknown_metric_fails_at_booster_create(built):
    from mmlspark_b200 import capi
    rng = np.random.default_rng(5)
    X = rng.standard_normal((2000, 4))
    ds = capi.Dataset.from_mat(X, DS_PARAMS).set_field("label", X[:, 0].astype(np.float32))
    with pytest.raises(capi.LightGBMError):
        capi.Booster(ds, BASE + "objective=regression metric=l2,not_a_metric")
