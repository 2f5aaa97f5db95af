"""The K1/K2 gradient kernels (csrc/objective.cuh), element by element, against independent numpy fp64 restatements of the LightGBM 3.2
objective formulas rounded to fp32, with the oracle's gradients as a second opinion.

Booster.get_gradients() returns the objective's gradients at the training scores.  Before the first iteration those are the training
set's init_score (an init_score turns boost-from-average off), so the init_score places every kernel at whatever input a case needs:
saturated sigmoids, logits of +-hundreds, exp close to the fp32 range, zero or huge weights, score == label, ties and -inf scores.

Point-wise kernels compute in fp64 and store fp32.  exp/log of CUDA and of the host may differ by an fp64 ulp and nvcc may contract
a*b+c into an FMA, so an element passes when |got - want| <= 1 fp32 ulp(want) + 2^-50 * (sum of |terms| before the final cancellation).
The lambdarank pair arithmetic has nothing to contract and its fp32 sums follow the reference's order: without lambdarank_norm it must
be bit-identical."""
import functools
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DS_PARAMS = "max_bin=63 is_pre_partition=True bin_construct_sample_cnt=50000 num_threads=0"
BASE = "num_leaves=7 learning_rate=0.1 min_data_in_leaf=20 verbosity=-1 "
N = (1 << 20) + 3          # the K1 grid is 8 blocks of 256 threads per SM: every thread makes several passes, the last one ragged


def _booster(y, init_score, params, weight=None, group=None, n_feat=2, seed=0):
    from mmlspark_b200 import capi
    n = len(y)
    X = np.random.default_rng(seed).standard_normal((n, n_feat))
    ds = capi.Dataset.from_mat(X, DS_PARAMS).set_field("label", y).set_field("init_score", init_score)
    if weight is not None:
        ds.set_field("weight", weight)
    if group is not None:
        ds.set_field("group", group)
    return capi.Booster(ds, BASE + params), ds, X


def _oracle(X, y, init_score, params, weight=None, group=None):
    from oracle import oracle as O
    ods = O.OracleDataset(X, DS_PARAMS).set_field("label", y).set_field("init_score", init_score)
    if weight is not None:
        ods.set_field("weight", weight)
    if group is not None:
        ods.set_field("group", group)
    ob = O.OracleBooster(ods, BASE + params)
    return ob.gradients()        # taken at the oracle's current scores: the init_score, before any update


def _exp(x):
    """exp rounded from extended precision (numpy's vectorised fp64 exp may be a few ulp off); overflows to inf like fp64"""
    with np.errstate(over="ignore"):
        return np.exp(np.asarray(x, dtype=np.longdouble)).astype(np.float64)


def _check(got, want64, terms, what):
    """got (fp32) against the fp64 reference want64 rounded to fp32; terms = sum of |terms| that cancel into want64"""
    want = np.asarray(want64, dtype=np.float64).astype(np.float32)
    assert np.isfinite(want).all(), what + ": the reference left the fp32 range"
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    bound = np.spacing(np.abs(want)).astype(np.float64) + 2.0 ** -50 * (np.abs(terms) + np.abs(want64))
    bad = np.nonzero(~(err <= bound))[0]
    differ = int(np.count_nonzero(got.view(np.uint32) != want.view(np.uint32)))
    print("%s: %d of %d elements not bit-identical" % (what, differ, got.size))
    assert bad.size == 0, "%s: %d elements off, first at %d: got %r want %r (fp64 %r)" % (
        what, bad.size, bad[0], got[bad[0]], want[bad[0]], want64[bad[0]])


def _weights(rng, n):
    w = rng.uniform(0.25, 4.0, n).astype(np.float32)
    w[::97] = 0.0
    w[1::89] = 1e-30
    w[2::83] = 1e6
    return w


# ---------------------------------------------------------------- restatements of LightGBM 3.2 ObjectiveFunction::GetGradients
def _pointwise(obj, s, y, w, p):
    """-> g64, h64, terms_g, terms_h (fp64; terms = what cancels).  p: the objective's parameters."""
    y = y.astype(np.float64)
    one = np.ones_like(s)
    wt = one if w is None else w.astype(np.float64)
    if obj == "regression":                                     # RegressionL2loss
        g, h, tg, th = s - y, one, np.abs(s) + np.abs(y), 0 * s
    elif obj == "huber":                                        # RegressionHuberLoss
        d = s - y
        g = np.where(np.abs(d) <= p["alpha"], d, np.sign(d) * p["alpha"])
        h, tg, th = one, np.abs(s) + np.abs(y), 0 * s
    elif obj == "fair":                                         # RegressionFairLoss
        c, x = p["fair_c"], s - y
        g, h = c * x / (np.abs(x) + c), c * c / ((np.abs(x) + c) * (np.abs(x) + c))
        tg = th = np.abs(s) + np.abs(y)
    elif obj == "poisson":                                      # RegressionPoissonLoss
        e = _exp(s)
        g, h, tg, th = e - y, _exp(s + p["poisson_max_delta_step"]), e + np.abs(y), 0 * s
    elif obj == "gamma":                                        # RegressionGammaLoss
        e = y * _exp(-s)
        g, h, tg, th = 1.0 - e, e, 1.0 + e, 0 * s
    elif obj == "tweedie":                                      # RegressionTweedieLoss
        rho = p["tweedie_variance_power"]
        e1, e2 = _exp((1 - rho) * s), _exp((2 - rho) * s)
        g, h = -y * e1 + e2, -y * (1 - rho) * e1 + (2 - rho) * e2
        tg, th = np.abs(y) * e1 + e2, np.abs(y * (1 - rho)) * e1 + (2 - rho) * e2
    elif obj == "cross_entropy":                                # CrossEntropy: z = 1 / (1 + exp(-s))
        z = 1.0 / (1.0 + _exp(-s))
        g, h, tg, th = z - y, z * (1.0 - z), z + np.abs(y), z * (1.0 + z)
    elif obj == "binary":                                       # BinaryLogloss: label_val {-1, 1}, label_weights {neg, pos}
        pos = y > 0
        npos, nneg = float(pos.sum()), float((~pos).sum())
        lw = [1.0, 1.0]
        if p.get("is_unbalance") and npos > 0 and nneg > 0:
            lw = [npos / nneg, 1.0] if npos > nneg else [1.0, nneg / npos]
        lw[1] *= p.get("scale_pos_weight", 1.0)
        sig, lab, lwv = p["sigmoid"], np.where(pos, 1.0, -1.0), np.where(pos, lw[1], lw[0])
        r = -lab * sig / (1.0 + _exp(lab * sig * s))
        ar = np.abs(r)
        g, h = r * lwv, ar * (sig - ar) * lwv
        tg, th = 0 * s, ar * (sig + ar) * lwv
    else:
        raise AssertionError(obj)
    if w is not None:
        g, h, tg, th = g * wt, h * wt, tg * wt, th * wt
    return g, h, tg, th


POINTWISE = [
    ("regression", "", {}),
    ("huber", "alpha=0.35", {"alpha": 0.35}),
    ("fair", "fair_c=2.3", {"fair_c": 2.3}),
    ("poisson", "poisson_max_delta_step=0.9", {"poisson_max_delta_step": 0.9}),
    ("gamma", "", {}),
    ("tweedie", "tweedie_variance_power=1.1", {"tweedie_variance_power": 1.1}),
    ("tweedie", "tweedie_variance_power=1.9", {"tweedie_variance_power": 1.9}),
    ("binary", "sigmoid=1", {"sigmoid": 1.0}),
    ("binary", "sigmoid=2.5 is_unbalance=true", {"sigmoid": 2.5, "is_unbalance": True}),
    ("binary", "sigmoid=2.5 scale_pos_weight=3.5", {"sigmoid": 2.5, "scale_pos_weight": 3.5}),
    ("cross_entropy", "", {}),
]


def _pointwise_data(obj, n, weighted, seed):
    rng = np.random.default_rng(seed)
    if obj in ("poisson", "gamma", "tweedie"):
        hi = 60.0 if weighted else 80.0                 # exp(|s|) times the label (and a 1e6 weight) stays inside fp32
        s = rng.uniform(-hi, hi, n)
        y = np.floor(rng.exponential(2.0, n)).astype(np.float32) if obj == "poisson" else rng.exponential(2.0, n).astype(np.float32)
        if obj == "gamma":
            y = np.maximum(y, np.float32(1e-3))
        s[:1000] = np.log(np.maximum(y[:1000], 1e-3).astype(np.float64))     # exp(s) close to the label: the gradient cancels
    elif obj == "binary":
        y = (rng.random(n) < 0.3).astype(np.float32)
        s = rng.uniform(-700, 700, n)                    # |sigmoid * s| far past the range of exp: saturated responses
        s[::3] = rng.normal(0, 3, s[::3].size)
    elif obj == "cross_entropy":
        y = rng.random(n).astype(np.float32)
        y[::4] = np.round(y[::4])                        # labels in {0, 1} and fractional
        s = rng.uniform(-40, 40, n)
        s[::3] = rng.normal(0, 2, s[::3].size)
    else:
        y = rng.normal(0, 10, n).astype(np.float32)
        s = y.astype(np.float64) + rng.normal(0, 1, n) * np.where(rng.random(n) < 0.5, 0.1, 30.0)
        s[::5] = y[::5]                                  # score == label exactly
    return s, y, (_weights(rng, n) if weighted else None)


@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("obj,params,p", POINTWISE, ids=["%s-%s" % (o, q.replace(" ", "-") or "default") for o, q, _ in POINTWISE])
def test_pointwise_gradients_match_fp64_reference(built, obj, params, p, weighted):
    s, y, w = _pointwise_data(obj, N, weighted, seed=len(obj) + 7 * weighted)
    b, _, _ = _booster(y, s, "objective=%s %s" % (obj, params), weight=w)
    got_g, got_h = b.get_gradients()
    g, h, tg, th = _pointwise(obj, s, y, w, p)
    _check(got_g, g, tg, obj + " grad")
    _check(got_h, h, th, obj + " hess")
    assert b.get_info()["constant_hessian"] is (obj == "regression" and not weighted)


@pytest.mark.parametrize("obj,params,p", POINTWISE, ids=["%s-%s" % (o, q.replace(" ", "-") or "default") for o, q, _ in POINTWISE])
def test_pointwise_gradients_match_oracle(built, obj, params, p):
    n = 6007
    s, y, w = _pointwise_data(obj, n, True, seed=3)
    b, _, X = _booster(y, s, "objective=%s %s" % (obj, params), weight=w)
    got_g, got_h = b.get_gradients()
    og, oh = _oracle(X, y, s, "objective=%s %s" % (obj, params), weight=w)
    g, h, tg, th = _pointwise(obj, s, y, w, p)
    _check(got_g, og.astype(np.float64), tg + np.abs(g), obj + " grad vs oracle")
    _check(got_h, oh.astype(np.float64), th + np.abs(h), obj + " hess vs oracle")


# ---------------------------------------------------------------- constant-hessian objectives: sign and percentile gradients
def _percentile_data(n, seed):
    rng = np.random.default_rng(seed)
    y = rng.normal(0, 5, n).astype(np.float32)
    y[::7] = rng.uniform(-0.9, 0.9, y[::7].size)       # |label| < 1: mape's label weight is 1
    s = y.astype(np.float64) + rng.normal(0, 2, n)
    s[::5] = y[::5]                                      # score == label: sign 0 (quantile: delta >= 0)
    # labels near 1e-30 and scores an fp64 ulp below: s - y < 0 in fp64 but rounds to -0 in fp32, where quantile counts delta >= 0
    y[3::101] = np.float32(1e-30)
    s[3::101] = np.nextafter(np.float64(np.float32(1e-30)), -np.inf)
    return s, y


@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("obj,params,alpha", [("regression", "", None), ("regression_l1", "", None), ("quantile", "alpha=0.1", 0.1),
                                              ("quantile", "alpha=0.9", 0.9), ("mape", "", None)])
def test_constant_hessian_objectives(built, obj, params, alpha, weighted):
    rng = np.random.default_rng(11)
    s, y = _percentile_data(N, 12)
    w = _weights(rng, N) if weighted else None
    b, _, _ = _booster(y, s, "objective=%s %s" % (obj, params), weight=w)
    assert b.get_info()["constant_hessian"] is (not weighted)
    got_g, got_h = b.get_gradients()
    w32 = np.ones(N, np.float32) if w is None else w
    np.testing.assert_array_equal(got_h, w32)                                  # exactly 1, or exactly the weight
    d = s - y.astype(np.float64)
    sgn = np.sign(d)
    if obj == "regression":
        g, tg = d * w32, (np.abs(s) + np.abs(y)) * w32
        _check(got_g, g, tg, obj + " grad")
        return
    if obj == "regression_l1":                                                 # Sign(diff) * weight
        want = (sgn * w32).astype(np.float32)
    elif obj == "quantile":                                                    # delta = score_t(s - y); alpha is a score_t
        a = np.float32(alpha)
        delta = d.astype(np.float32)
        want = np.where(delta >= 0, np.float32(1) - a, -a).astype(np.float32)
        if w is not None:
            want = want * w
        assert (d[3::101] < 0).all() and (delta[3::101] == 0).all()
    else:                                                                      # mape: label_weight = 1 / max(1, |label|) (* weight)
        lw = np.float32(1) / np.maximum(np.float32(1), np.abs(y))
        if w is not None:
            lw = lw * w
        want = (sgn * lw.astype(np.float64)).astype(np.float32)
    np.testing.assert_array_equal(got_g, want)


# ---------------------------------------------------------------- multiclass
def _softmax_grads(S, lab, w):
    """MulticlassSoftmax::GetGradients with Common::Softmax (max shift, sequential sum over the classes); S: [K][n]"""
    K = S.shape[0]
    wmax = S[0].copy()
    for k in range(1, K):
        wmax = np.maximum(wmax, S[k])
    e = [_exp(S[k] - wmax) for k in range(K)]
    wsum = np.zeros_like(wmax)
    for k in range(K):
        wsum = wsum + e[k]
    factor = K / (K - 1.0)
    G, H, TG, TH = [], [], [], []
    wt = 1.0 if w is None else w.astype(np.float64)
    for k in range(K):
        pk = e[k] / wsum
        G.append(np.where(lab == k, pk - 1.0, pk) * wt)
        H.append(factor * pk * (1.0 - pk) * wt)
        TG.append(np.where(lab == k, pk + 1.0, 0.0) * wt)
        TH.append(factor * pk * (1.0 + pk) * wt)
    return [np.concatenate(a) for a in (G, H, TG, TH)]


@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("K", [3, 30])
def test_multiclass_softmax(built, K, weighted):
    n = N if K == 3 else (1 << 19) + 3
    rng = np.random.default_rng(K)
    lab = rng.integers(0, K, n)
    S = rng.normal(0, 4, (K, n))
    big = rng.random(n) < 0.2
    S[:, big] = rng.uniform(-800, 800, (K, int(big.sum())))     # exp of the unshifted logits overflows / underflows fp64
    low = rng.random(n) < 0.05
    S[:, low] = rng.uniform(-800, -750, (K, int(low.sum())))     # every class far below 0
    S[:, 1::17] = 5.0                                            # all classes tied
    w = _weights(rng, n) if weighted else None
    b, _, _ = _booster(lab.astype(np.float32), S.ravel(), "objective=multiclass num_class=%d" % K, weight=w)
    got_g, got_h = b.get_gradients()
    g, h, tg, th = _softmax_grads(S, lab, w)
    _check(got_g, g, tg, "softmax K=%d grad" % K)
    _check(got_h, h, th, "softmax K=%d hess" % K)


@pytest.mark.parametrize("unbalance", [False, True], ids=["balanced", "is_unbalance"])
def test_multiclassova(built, unbalance):
    """One BinaryLogloss per class on (label == k); class 2 has no positive row: it is not trained, its gradients stay 0 and its
    trees are constant."""
    from mmlspark_b200.modeltext import parse_model
    K, n, sig = 4, N, 1.7
    rng = np.random.default_rng(41)
    lab = rng.choice([0, 1, 3], n, p=[0.6, 0.3, 0.1])
    S = rng.uniform(-500, 500, (K, n))
    S[:, ::2] = rng.normal(0, 2, (K, S[:, ::2].shape[1]))
    params = "objective=multiclassova num_class=%d sigmoid=%g scale_pos_weight=1.5%s" % (K, sig, " is_unbalance=true" if unbalance else "")
    b, _, _ = _booster(lab.astype(np.float32), S.ravel(), params)
    got_g, got_h = b.get_gradients()
    for k in range(K):
        seg = slice(k * n, (k + 1) * n)
        if k == 2:
            assert not got_g[seg].any() and not got_h[seg].any()
            continue
        y = (lab == k).astype(np.float32)
        g, h, tg, th = _pointwise("binary", S[k], y, None, {"sigmoid": sig, "is_unbalance": unbalance, "scale_pos_weight": 1.5})
        _check(got_g[seg], g, tg, "ova class %d grad" % k)
        _check(got_h[seg], h, th, "ova class %d hess" % k)
    for _ in range(2):
        b.update_one_iter()
    trees = parse_model(b.save_model_to_string())["trees"]
    assert len(trees) == 2 * K
    for t, tree in enumerate(trees):
        assert (tree["num_leaves"] == 1) == (t % K == 2), "tree %d" % t


# ---------------------------------------------------------------- lambdarank
@functools.lru_cache(maxsize=4)
def _sigmoid_table(sigmoid):
    """LambdarankNDCG's 1M-entry table of 1 / (1 + exp(sigmoid * x)) over x in [-50 / sigmoid / 2, 50 / sigmoid / 2], stored as score_t"""
    bins = 1 << 20
    min_in = -50.0 / sigmoid / 2
    max_in = -min_in
    factor = bins / (max_in - min_in)
    tab = np.array([1.0 / (1.0 + math.exp((i / factor + min_in) * sigmoid)) for i in range(bins)], dtype=np.float64).astype(np.float32)
    return tab, min_in, max_in, factor


def _default_gain():
    return np.array([0.0] + [float((1 << i) - 1) for i in range(1, 31)])


def _lambdarank_query(s, y, trunc, norm, sigmoid, gain, disc):
    """LambdarankNDCG::GetGradientsForOneQuery for one query (before weights), vectorised over the pairs (i, j), i < min(truncation,
    cnt - 1), j > i, of the stable descending order; every document's fp32 lambda / hessian is summed in the reference's pair order"""
    cnt = len(s)
    lam, hes = np.zeros(cnt, np.float32), np.zeros(cnt, np.float32)
    li = y.astype(np.int64)
    # DCGCalculator::CalMaxDCGAtK(truncation): the best labels first
    lc = np.bincount(li, minlength=len(gain))
    top, maxdcg = len(gain) - 1, 0.0
    for j in range(min(trunc, cnt)):
        while top > 0 and lc[top] <= 0:
            top -= 1
        maxdcg += disc[j] * gain[top]
        lc[top] -= 1
    imd = 1.0 / maxdcg if maxdcg > 0 else maxdcg
    order = np.argsort(-s, kind="stable")
    ss, ls = s[order], li[order]
    teff = min(trunc, cnt - 1)
    if teff <= 0:
        return lam, hes
    best = ss[0]
    worst_idx = cnt - 1
    if worst_idx > 0 and ss[worst_idx] == -np.inf:
        worst_idx -= 1
    worst = ss[worst_idx]
    I, J = np.arange(teff)[:, None], np.arange(cnt)[None, :]
    valid = (J > I) & (ss[I] != -np.inf) & (ss[J] != -np.inf) & (ls[I] != ls[J])
    i_high = ls[I] > ls[J]
    hr, lr = np.where(i_high, I, J), np.where(i_high, J, I)
    with np.errstate(invalid="ignore"):
        ds = np.where(valid, ss[hr] - ss[lr], 0.0)
    delta = (gain[ls[hr]] - gain[ls[lr]]) * np.abs(disc[hr] - disc[lr]) * imd
    if norm and best != worst:
        delta = delta / (np.float64(np.float32(0.01)) + np.abs(ds))
    tab, min_in, max_in, factor = _sigmoid_table(sigmoid)
    raw = np.clip((ds - min_in) * factor, 0, len(tab) - 1)
    idx = np.where(ds <= min_in, 0, np.where(ds >= max_in, len(tab) - 1, raw.astype(np.int64)))
    pl = tab[idx].astype(np.float64)
    ph = pl * (1.0 - pl)
    pl = pl * (-sigmoid * delta)
    ph = ph * (sigmoid * sigmoid * delta)
    pl, ph = np.where(valid, pl, 0.0), np.where(valid, ph, 0.0)
    fl, fh = pl.astype(np.float32), ph.astype(np.float32)
    # lambdas[high] += p_lambda, lambdas[low] -= p_lambda.  Document p meets (0, p) .. (p - 1, p) first (as j), then (p, p + 1) ..
    # (p, cnt - 1) (as i).  Zero entries for the skipped pairs leave an fp32 sum unchanged.
    as_j = np.add.accumulate(np.where(i_high, -fl, fl), axis=0, dtype=np.float32)[-1]
    hs_j = np.add.accumulate(fh, axis=0, dtype=np.float32)[-1]
    as_i = np.add.accumulate(np.concatenate([as_j[:teff, None], np.where(i_high, fl, -fl)], axis=1), axis=1, dtype=np.float32)[:, -1]
    hs_i = np.add.accumulate(np.concatenate([hs_j[:teff, None], fh], axis=1), axis=1, dtype=np.float32)[:, -1]
    lam_s, hes_s = as_j.copy(), hs_j.copy()
    lam_s[:teff], hes_s[:teff] = as_i, hs_i
    if norm:
        sum_lambdas = float(np.sum(-2.0 * pl[valid]))
        if sum_lambdas > 0:
            nf = math.log2(1 + sum_lambdas) / sum_lambdas
            lam_s = (lam_s.astype(np.float64) * nf).astype(np.float32)
            hes_s = (hes_s.astype(np.float64) * nf).astype(np.float32)
    lam[order], hes[order] = lam_s, hes_s
    return lam, hes


def _lambdarank_reference(s, y, sizes, w, trunc, norm, sigmoid=1.0, gain=None):
    gain = _default_gain() if gain is None else np.asarray(gain, dtype=np.float64)
    disc = np.array([1.0 / math.log2(2.0 + i) for i in range(int(max(sizes)) + 1)])      # DCGCalculator's discount table
    g, h = np.zeros(len(s), np.float32), np.zeros(len(s), np.float32)
    off = 0
    for c in sizes:
        sl = slice(off, off + c)
        g[sl], h[sl] = _lambdarank_query(s[sl], y[sl], trunc, norm, sigmoid, gain, disc)
        off += c
    if w is not None:                                                              # score_t * label_t
        g, h = g * w, h * w
    return g, h


SIZES = [1, 2, 31, 32, 33, 95, 96, 97, 127, 128, 129, 300, 1000]


def _ranking_data(seed, max_label=30, gain_len=31):
    """every size of SIZES with random scores, then the edge queries: all scores tied, scores rounded to 0.5, a few -inf scores,
    all labels equal, a single relevant document"""
    rng = np.random.default_rng(seed)
    sizes = SIZES + [200, 150, 140, 97, 129]
    n = sum(sizes)
    y = rng.integers(0, min(max_label, gain_len - 1) + 1, n).astype(np.float32)
    y[rng.random(n) < 0.5] = 0
    s = rng.normal(0, 3, n)
    off = np.cumsum([0] + sizes)
    q = len(SIZES)
    s[off[q]:off[q + 1]] = 0.0                                               # all tied: the scores of iteration 0
    s[off[q + 1]:off[q + 2]] = np.round(2 * rng.normal(0, 1, sizes[q + 1])) / 2
    r = slice(off[q + 2], off[q + 3])
    s[r][rng.choice(sizes[q + 2], 7, replace=False)] = -np.inf                # -inf scores: skipped pairs and the worst_idx step
    y[off[q + 3]:off[q + 4]] = 3                                             # all labels equal: no pair
    y[off[q + 4]:off[q + 5]] = 0
    y[off[q + 4] + 77] = 2                                                   # one relevant document
    return s, y, np.array(sizes, dtype=np.int32)


@pytest.mark.parametrize("norm", [False, True], ids=["no_norm", "norm"])
@pytest.mark.parametrize("trunc", [1, 30, 48, 64, 180])
def test_lambdarank_gradients(built, trunc, norm):
    s, y, sizes = _ranking_data(trunc)
    params = "objective=lambdarank lambdarank_truncation_level=%d lambdarank_norm=%s" % (trunc, "true" if norm else "false")
    b, _, _ = _booster(y, s, params, group=sizes)
    got_g, got_h = b.get_gradients()
    want_g, want_h = _lambdarank_reference(s, y, sizes, None, trunc, norm)
    assert np.isfinite(want_g).all() and np.abs(want_g).max() > 0
    if norm:
        np.testing.assert_allclose(got_g, want_g, rtol=1e-6, atol=0)      # sum_lambdas is summed in another order
        np.testing.assert_allclose(got_h, want_h, rtol=1e-6, atol=0)
    else:
        np.testing.assert_array_equal(got_g, want_g)
        np.testing.assert_array_equal(got_h, want_h)


@pytest.mark.parametrize("norm", [False, True], ids=["no_norm", "norm"])
def test_lambdarank_weights_sigmoid_and_oracle(built, norm):
    s, y, sizes = _ranking_data(5)
    w = np.random.default_rng(6).uniform(0.1, 3.0, len(y)).astype(np.float32)
    params = "objective=lambdarank lambdarank_truncation_level=30 sigmoid=1.7 lambdarank_norm=%s" % ("true" if norm else "false")
    b, _, X = _booster(y, s, params, weight=w, group=sizes)
    got_g, got_h = b.get_gradients()
    want_g, want_h = _lambdarank_reference(s, y, sizes, w, 30, norm, sigmoid=1.7)
    og, oh = _oracle(X, y, s, params, weight=w, group=sizes)
    if norm:
        for a, bb in ((got_g, want_g), (got_h, want_h), (got_g, og), (got_h, oh)):
            np.testing.assert_allclose(a, bb, rtol=1e-6, atol=0)
    else:
        for a, bb in ((got_g, want_g), (got_h, want_h), (got_g, og), (got_h, oh)):
            np.testing.assert_array_equal(a, bb)


def test_lambdarank_long_label_gain(built):
    """a custom label_gain of 100 entries with labels up to 99"""
    gain = np.round(np.linspace(0.0, 50.0, 100) ** 1.5, 3)
    s, y, sizes = _ranking_data(8, max_label=99, gain_len=100)
    params = "objective=lambdarank lambdarank_truncation_level=64 lambdarank_norm=false label_gain=" + ",".join(repr(float(v)) for v in gain)
    b, _, _ = _booster(y, s, params, group=sizes)
    got_g, got_h = b.get_gradients()
    want_g, want_h = _lambdarank_reference(s, y, sizes, None, 64, False, gain=gain)
    np.testing.assert_array_equal(got_g, want_g)
    np.testing.assert_array_equal(got_h, want_h)


# k_grad_lambdarank keeps one query in shared memory: 32 bytes per document plus the pair matrix of one j-tile, truncation x (tile + 1)
# float2.  At truncation 180 the tile is 32 documents and 200 KB hold 4914 documents.
_LIMIT_180 = (200 * 1024 - 8 - 180 * 33 * 8) // 32


def test_lambdarank_query_at_shared_memory_limit(built):
    rng = np.random.default_rng(12)
    sizes = np.array([_LIMIT_180, 40], dtype=np.int32)
    n = int(sizes.sum())
    y = rng.integers(0, 6, n).astype(np.float32)
    s = np.round(rng.normal(0, 2, n), 1)
    b, _, _ = _booster(y, s, "objective=lambdarank lambdarank_truncation_level=180 lambdarank_norm=false", group=sizes)
    got_g, got_h = b.get_gradients()
    want_g, want_h = _lambdarank_reference(s, y, sizes, None, 180, False)
    np.testing.assert_array_equal(got_g, want_g)
    np.testing.assert_array_equal(got_h, want_h)


def test_lambdarank_query_above_shared_memory_limit_is_rejected(built):
    from mmlspark_b200 import capi
    n = _LIMIT_180 + 1
    y = (np.arange(n) % 3).astype(np.float32)
    with pytest.raises(capi.LightGBMError, match="too large for the lambdarank kernel"):
        _booster(y, np.zeros(n), "objective=lambdarank lambdarank_truncation_level=180", group=np.array([n], dtype=np.int32))


def test_lambdarank_rejects_fractional_label(built):
    from mmlspark_b200 import capi
    y = np.array([0, 1, 1.5, 2] * 10, dtype=np.float32)
    with pytest.raises(capi.LightGBMError, match="label should be int type"):
        _booster(y, np.zeros(len(y)), "objective=lambdarank", group=np.array([len(y)], dtype=np.int32))


# ---------------------------------------------------------------- the accessor changes nothing
@pytest.mark.parametrize("params", ["objective=binary", "objective=multiclass num_class=3", "objective=regression boosting=rf bagging_freq=1 bagging_fraction=0.5",
                                    "objective=lambdarank"])
def test_get_gradients_is_inert(built, params):
    from mmlspark_b200 import capi
    rng = np.random.default_rng(21)
    n = 6000
    X = rng.standard_normal((n, 5))
    y = (np.clip(np.round(X[:, 0] + 1.5), 0, 2) if ("multiclass" in params or "lambdarank" in params) else (X[:, 0] > 0)).astype(np.float32)
    models = []
    for probe in (False, True):
        ds = capi.Dataset.from_mat(X, DS_PARAMS).set_field("label", y)
        if "lambdarank" in params:
            ds.set_field("group", np.full(n // 20, 20, dtype=np.int32))
        b = capi.Booster(ds, BASE + params)
        for _ in range(3):
            if probe:
                before = b.get_scores(0)
                g, h = b.get_gradients()
                assert np.isfinite(g).all() and np.isfinite(h).all() and g.any()
                np.testing.assert_array_equal(b.get_scores(0), before)
            b.update_one_iter()
        models.append(b.save_model_to_string())
    assert models[0] == models[1]
