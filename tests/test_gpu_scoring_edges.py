"""GPU parity tests for the scoring path at its edges: one-vs-one SVC up to the 32-class limit (pair enumeration, per-pair
class weights, votes, dual_coef_ layout, decision values over more than one column block), every fused classification
scorer on general splitters, absent classes, label encodings, roc_auc ties and single-class test sets, the multinomial
LogisticRegression limit, and the regression scorers of Lasso / ElasticNet including constant-target test sets.

Every comparison is between values that must be equal, and each test proves that in its own body:
  * SVC follows scikit-learn's SMO trajectory exactly.  Predictions are compared at 1e-12 after asserting, from
    scikit-learn's own fits, that no scored prediction hinges on a decision value within DELTA_SVC of zero (a last-bit
    difference of the float32 kernel matrix, CUDA's exp against the host's, could move such a value across zero).
  * LogisticRegression is float32-faithful, not bit-exact.  Every scored row's |z| (binary) or top-two logit gap
    (multinomial) in scikit-learn's fit is asserted to be at least DELTA_LOGREG, so count-based scores must be equal.
  * roc_auc may differ by the pairs whose scikit-learn scores lie closer than the margin without being equal (for SVC,
    DELTA_SVC: predictions are exact, but a decision value may move by less than the margin).
The scikit-learn references are the per-split fits GridSearchCV makes (clone, fit on the training rows, score on the
test / training rows); each is fitted once and then scored with every scorer."""
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# Scored one-vs-one decision values of the SVC data below stay at least this far from zero, or their sign cannot change
# the vote (checked per test).
DELTA_SVC = 1e-3
# LogisticRegression margins, calibrated once on a CPU against the float32-faithful restatement of the fit
# (oracle.logreg_fit_score's optimiser) on the data below.  Binary: |z| differs from scikit-learn's by at most 1.0e-6; the
# margin is 1e-3, which also leaves room for the device's early stop moving by an iteration between runs (its loss sum
# uses floating-point atomics), a move this calibration does not see.  Multinomial, C <= 0.01: the top-two logit gap
# differs by at most 1.1e-3 (K = 5, and 9.0e-4 on the absent-class data) and 8.0e-2 (K = 64); the margins are about 10x.
DELTA_LOGREG = 1e-3
DELTA_LOGREG_MULTI = {5: 1.2e-2, 64: 0.9}

CLASSIFICATION_SCORERS = ["accuracy", "balanced_accuracy", "f1", "precision", "recall", "roc_auc", "f1_macro",
                          "f1_micro", "f1_weighted"]
MULTICLASS_SCORERS = ["accuracy", "balanced_accuracy", "f1_macro", "f1_micro", "f1_weighted"]


# ------------------------------------------------------------------ data -------------------------
def _blobs(n_per_class, k, d, seed, std=1.0, box=6.0):
    """k Gaussian blobs of unequal sizes (so the averaged scorers differ), float32"""
    from sklearn.datasets import make_blobs
    X, y = make_blobs(n_samples=list(n_per_class), n_features=d, cluster_std=std, center_box=(-box, box),
                      random_state=seed)
    return X.astype(np.float32), y


def _svc12():
    # Seed 0 of 0-3: every prediction of the 25 fits below is certified at DELTA_SVC (seed 2 is not).
    k, n = 12, 5000
    sizes = [n // k + (i - k // 2) * 25 for i in range(k)]
    sizes[-1] += n - sum(sizes)
    return _blobs(sizes, k, 8, seed=0)


def _gap_binary(n, d, seed, flip=0.08, gap=1.0):
    """Two classes on either side of a hyperplane with no row within `gap` of it, and a fraction of labels flipped
    (misclassified rows far from the boundary): non-trivial scores with every row far from the fitted boundary."""
    rng = np.random.RandomState(seed)
    X = rng.randn(4 * n, d)
    w = rng.randn(d)
    s = X @ w / np.linalg.norm(w)
    keep = np.flatnonzero(np.abs(s) > gap)[:n]
    X, y = X[keep], (s[keep] > 0).astype(int)
    f = rng.rand(n) < flip
    y[f] = 1 - y[f]
    return X.astype(np.float32), y


# ------------------------------------------------------------------ references -------------------
def _metric(name):
    from sklearn import metrics as M
    return {"accuracy": M.accuracy_score,
            "balanced_accuracy": M.balanced_accuracy_score,
            "f1": lambda t, p: M.f1_score(t, p, pos_label=1),
            "precision": lambda t, p: M.precision_score(t, p, pos_label=1),
            "recall": lambda t, p: M.recall_score(t, p, pos_label=1),
            "f1_macro": lambda t, p: M.f1_score(t, p, average="macro"),
            "f1_micro": lambda t, p: M.f1_score(t, p, average="micro"),
            "f1_weighted": lambda t, p: M.f1_score(t, p, average="weighted")}[name]


class _Fits:
    """scikit-learn's per-split fits of a candidate list: predictions and decision values of every row."""

    def __init__(self, est, cands, X, y, splits, ovo=False):
        from sklearn.base import clone
        self.X, self.y, self.splits, self.cands = X, np.asarray(y), splits, cands
        self.pred, self.dec, self.n_iter = {}, {}, {}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for ci, p in enumerate(cands):
                for k, (tr, te) in enumerate(splits):
                    m = clone(est).set_params(**p)
                    if ovo:
                        m.set_params(decision_function_shape="ovo")
                    m.fit(X[tr], self.y[tr])
                    self.pred[ci, k] = m.predict(X)
                    self.dec[ci, k] = m.decision_function(X)
                    self.n_iter[ci, k] = int(np.sum(getattr(m, "n_iter_", 0)))

    def rows(self, k, part):
        tr, te = self.splits[k]
        return te if part == "test" else tr

    def score(self, scoring, ci, k, part):
        r = self.rows(k, part)
        yt = self.y[r]
        if scoring == "roc_auc":
            from sklearn.metrics import roc_auc_score
            if len(np.unique(yt)) < 2:
                return np.nan                                      # roc_auc_score raises; error_score=nan
            return roc_auc_score(yt, self.dec[ci, k][r])
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return _metric(scoring)(yt, self.pred[ci, k][r])

    def auc_slack(self, ci, k, part, delta):
        """(pairs of opposite-label rows whose scores differ by less than delta but are not equal) / all such pairs"""
        r = self.rows(k, part)
        yt, s = self.y[r], self.dec[ci, k][r]
        lab = np.unique(yt)
        if len(lab) < 2:
            return 0.0
        sp, sn = s[yt == lab[1]], s[yt == lab[0]]
        diff = np.abs(sp[:, None] - sn[None, :])
        return np.count_nonzero((diff > 0) & (diff < delta)) / diff.size


def _vote_uncertain(dv, k, delta):
    """Rows whose one-vs-one vote could change if every decision value within delta of zero took the other sign
    (libsvm: dec > 0 votes for the lower class of the pair, the first maximum wins)."""
    n = len(dv)
    if k == 2:
        return np.abs(dv.reshape(n)) < delta
    votes, win_u, lose_u = np.zeros((n, k), int), np.zeros((n, k), int), np.zeros((n, k), int)
    p = 0
    for a in range(k):
        for b in range(a + 1, k):
            pos, unc = dv[:, p] > 0, np.abs(dv[:, p]) < delta
            votes[pos, a] += 1
            votes[~pos, b] += 1
            win_u[pos & unc, a] += 1
            win_u[~pos & unc, b] += 1
            lose_u[pos & unc, b] += 1
            lose_u[~pos & unc, a] += 1
            p += 1
    r = np.arange(n)
    pred = votes.argmax(1)
    lo = votes[r, pred] - win_u[r, pred]                           # fewest votes the winner can end with
    hi = votes + lose_u                                            # most votes any other class can reach
    hi[r, pred] = -1
    return ~(lo > hi.max(1)) & (np.abs(dv) < delta).any(1)        # a tied vote without such a value is deterministic


def _assert_svc_margin(ref, k_classes):
    for (ci, k), dv in ref.dec.items():
        tr, te = ref.splits[k]
        scored = np.concatenate([tr, te])
        bad = _vote_uncertain(dv[scored], k_classes, DELTA_SVC)
        assert not bad.any(), "candidate %d split %d: %d scored rows within %g of a vote change" % (ci, k, bad.sum(), DELTA_SVC)


def _assert_logreg_margin(ref, k_classes=2):
    for (ci, k), z in ref.dec.items():
        tr, te = ref.splits[k]
        z = z[np.concatenate([tr, te])]
        if z.ndim == 1:
            m, delta = np.abs(z), DELTA_LOGREG
        else:
            top = np.sort(z, 1)
            m, delta = top[:, -1] - top[:, -2], DELTA_LOGREG_MULTI[64 if k_classes > 5 else 5]
        assert m.min() >= delta, "candidate %d split %d: margin %.3g < %g" % (ci, k, m.min(), delta)


def _search(est, grid, X, y, cv, scoring, **kw):
    from spark_sklearn_b200 import GridSearchCV
    kw.setdefault("refit", False)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return GridSearchCV(None, est, grid, cv=cv, scoring=scoring, iid=False, **kw).fit(X, y)


def _assert_scores(a, ref, scoring, atol=1e-12, auc_delta=None):
    for ci in range(len(ref.cands)):
        for k in range(len(ref.splits)):
            for part in ("test", "train"):
                got = a.cv_results_["split%d_%s_score" % (k, part)][ci]
                want = ref.score(scoring, ci, k, part)
                tol = atol + (ref.auc_slack(ci, k, part, auc_delta) if scoring == "roc_auc" and auc_delta else 0.0)
                if np.isnan(want):
                    assert np.isnan(got), (scoring, ci, k, part, got)
                else:
                    assert abs(got - want) <= tol, (scoring, ci, k, part, got, want, tol)


def _grid_cands(grid):
    from sklearn.model_selection import ParameterGrid
    return list(ParameterGrid(grid))


# ------------------------------------------------------------------ 1. many-class SVC -------------
SVC12_GRID = [{"kernel": ["rbf"], "C": [1.0, 10.0], "gamma": [0.05, 0.2]}, {"kernel": ["linear"], "C": [0.5]}]


@pytest.fixture(scope="module")
def svc12():
    from sklearn.model_selection import StratifiedKFold
    from sklearn.svm import SVC
    X, y = _svc12()
    splits = list(StratifiedKFold(5).split(X, y))
    ref = _Fits(SVC(), _grid_cands(SVC12_GRID), X, y, splits, ovo=True)
    _assert_svc_margin(ref, 12)
    return X, y, splits, ref


@pytest.mark.parametrize("scoring", MULTICLASS_SCORERS)
def test_svc_12_classes_scorers_bitexact(engine, svc12, scoring):
    """12 classes, 66 pairs: 660 decision columns per gamma group (gridDim.y = 7 column blocks), n = 5000 >= 4096 so the
    support-row range is split into slabs."""
    from sklearn.model_selection import StratifiedKFold
    from sklearn.svm import SVC
    X, y, splits, ref = svc12
    a = _search(SVC(), SVC12_GRID, X, y, StratifiedKFold(5), scoring)
    _assert_scores(a, ref, scoring)


def test_svc_12_classes_n_iter_and_refit(engine, svc12):
    from oracle import oracle as O
    from sklearn.model_selection import StratifiedKFold
    from sklearn.svm import SVC
    X, y, splits, ref = svc12
    fold_id, ns = O.folds_from_cv(StratifiedKFold(5), X, y, True)
    engine.set_data(X, fold_id, ns, y_class=y.astype(np.int32))
    cands = ref.cands
    r = engine.svc([p["kernel"] for p in cands], [p["C"] for p in cands], [p.get("gamma", 0.0) for p in cands])
    it_ref = np.array([[ref.n_iter[ci, k] for k in range(ns)] for ci in range(len(cands))])
    assert np.mean(r["n_iter"] == it_ref) >= 0.97, (r["n_iter"], it_ref)     # iterations summed over the 66 pairs
    for ci in range(len(cands)):
        for k in range(ns):
            assert r["test"][ci, k] == ref.score("accuracy", ci, k, "test")
            assert r["train"][ci, k] == ref.score("accuracy", ci, k, "train")

    a = _search(SVC(), SVC12_GRID, X, y, StratifiedKFold(5), None, refit=True)
    means = np.array([np.mean([ref.score("accuracy", ci, k, "test") for k in range(ns)]) for ci in range(len(cands))])
    assert a.best_params_ == cands[int(np.argmax(means))]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sk = SVC(decision_function_shape="ovo").set_params(**a.best_params_).fit(X, y)
    dv = sk.decision_function(X)
    assert not _vote_uncertain(dv, 12, DELTA_SVC).any()
    ea = a.best_estimator_
    np.testing.assert_array_equal(ea.support_, sk.support_)
    np.testing.assert_array_equal(ea.n_support_, sk.n_support_)
    np.testing.assert_allclose(ea.dual_coef_, sk.dual_coef_, rtol=0, atol=1e-12)
    np.testing.assert_allclose(ea.intercept_, sk.intercept_, rtol=0, atol=1e-12)
    np.testing.assert_array_equal(a.predict(X), sk.predict(X))
    ea.set_params(decision_function_shape="ovo")
    np.testing.assert_allclose(ea.decision_function(X), dv, rtol=0, atol=1e-10)
    ea.set_params(decision_function_shape="ovr")
    sk.set_params(decision_function_shape="ovr")
    np.testing.assert_allclose(ea.decision_function(X), sk.decision_function(X), rtol=0, atol=1e-10)


def test_svc_12_classes_class_weight(engine, svc12):
    """Per-pair C x class_weight (weighted_C) with a dict that touches middle classes, and 'balanced' per training fold."""
    from sklearn.model_selection import StratifiedKFold
    from sklearn.svm import SVC
    X, y, splits, _ = svc12
    grid = {"C": [10.0], "gamma": [0.05], "class_weight": [{4: 3.0, 7: 0.25}, "balanced"]}
    ref = _Fits(SVC(), _grid_cands(grid), X, y, splits, ovo=True)
    _assert_svc_margin(ref, 12)
    for scoring in ("accuracy", "balanced_accuracy"):
        a = _search(SVC(), grid, X, y, StratifiedKFold(5), scoring)
        _assert_scores(a, ref, scoring)


def _svc32(k):
    # 32 classes of 24-33 rows in 8 dimensions, far apart: seed 1 certifies every prediction at DELTA_SVC
    return _blobs([24 + (i * 7) % 10 for i in range(k)], k, 8, seed=1, std=1.0, box=12.0)


def test_svc_32_classes_limit(engine):
    """The 32-class limit: 496 pairs per fit, the widest vote."""
    from sklearn.model_selection import StratifiedKFold
    from sklearn.svm import SVC
    X, y = _svc32(32)
    grid = {"C": [1.0, 10.0], "gamma": [0.02]}
    splits = list(StratifiedKFold(3).split(X, y))
    ref = _Fits(SVC(), _grid_cands(grid), X, y, splits, ovo=True)
    _assert_svc_margin(ref, 32)
    for scoring in ("f1_macro", "balanced_accuracy"):
        _assert_scores(_search(SVC(), grid, X, y, StratifiedKFold(3), scoring), ref, scoring)
    a = _search(SVC(), grid, X, y, StratifiedKFold(3), "accuracy", refit=True)
    _assert_scores(a, ref, "accuracy")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sk = SVC(decision_function_shape="ovo").set_params(**a.best_params_).fit(X, y)
    assert not _vote_uncertain(sk.decision_function(X), 32, DELTA_SVC).any()
    np.testing.assert_array_equal(a.predict(X), sk.predict(X))
    np.testing.assert_array_equal(a.best_estimator_.n_support_, sk.n_support_)
    np.testing.assert_allclose(a.best_estimator_.dual_coef_, sk.dual_coef_, rtol=0, atol=1e-12)


def test_svc_33_classes_raises(engine):
    from sklearn.svm import SVC
    from spark_sklearn_b200 import GridSearchCV
    from spark_sklearn_b200.engine import EngineError
    X, y = _svc32(33)
    gs = GridSearchCV(None, SVC(), {"C": [1.0]}, cv=3)
    with pytest.raises(EngineError, match="2..32 classes"):
        gs.fit(X, y)


# ------------------------------------------------------------------ 2. count-based scorer edges --
def _rare_class_data(k):
    """k - 1 blob classes plus a class of 3 rows: under StratifiedKFold(5) two test sets lack it"""
    X, y = _blobs([150] * (k - 1) + [3], k, 6, seed=3, std=1.0, box=10.0)
    return X, y


def _absent_class_cases(k):
    from sklearn.model_selection import PredefinedSplit, StratifiedKFold
    X, y = _rare_class_data(k)
    n = len(y)
    fold = np.arange(n) % 4
    fold[y == k - 2] = -1                                          # a class that only ever trains
    return X, y, {"stratified_rare": StratifiedKFold(5), "predefined_train_only": PredefinedSplit(fold)}


def _assert_absent_class_exercised(ref, k_classes):
    """At least one test set neither holds nor is predicted some class (else the case tests nothing)."""
    hit = False
    for (ci, k), pred in ref.pred.items():
        te = ref.splits[k][1]
        present = set(ref.y[te]) | set(pred[te])
        hit |= len(present) < k_classes
    assert hit


@pytest.mark.parametrize("case,k_classes", [("stratified_rare", 2), ("stratified_rare", 4), ("predefined_train_only", 4)])
def test_svc_absent_class_scorers(engine, case, k_classes):
    from sklearn.svm import SVC
    X, y, cvs = _absent_class_cases(k_classes)
    kc = len(np.unique(y))
    cv = cvs[case]
    grid = {"C": [1.0, 10.0], "gamma": [0.05]}
    ref = _Fits(SVC(), _grid_cands(grid), X, y, list(cv.split(X, y)), ovo=True)
    _assert_svc_margin(ref, kc)
    _assert_absent_class_exercised(ref, kc)
    for scoring in MULTICLASS_SCORERS:
        a = _search(SVC(), grid, X, y, cv, scoring)
        _assert_scores(a, ref, scoring)


@pytest.mark.parametrize("case,k_classes", [("stratified_rare", 2), ("stratified_rare", 4), ("predefined_train_only", 4)])
def test_logreg_absent_class_scorers(engine, case, k_classes):
    from sklearn.linear_model import LogisticRegression
    X, y, cvs = _absent_class_cases(k_classes)
    kc = len(np.unique(y))
    cv = cvs[case]
    grid = {"C": [0.002, 0.01]}
    ref = _Fits(LogisticRegression(), _grid_cands(grid), X, y, list(cv.split(X, y)))
    _assert_logreg_margin(ref, kc)
    _assert_absent_class_exercised(ref, kc)
    for scoring in MULTICLASS_SCORERS:
        a = _search(LogisticRegression(), grid, X, y, cv, scoring)
        _assert_scores(a, ref, scoring)


def _general_cvs(y):
    from sklearn.model_selection import PredefinedSplit, RepeatedStratifiedKFold, StratifiedShuffleSplit
    n = len(y)
    pre = np.arange(n) % 4
    pre[: n // 5] = -1
    return {"shuffle": StratifiedShuffleSplit(4, test_size=0.25, train_size=0.5, random_state=5),
            "repeated": RepeatedStratifiedKFold(n_splits=3, n_repeats=2, random_state=5),
            "predefined": PredefinedSplit(pre)}


@pytest.fixture(scope="module")
def gap_binary():
    return _gap_binary(1200, 10, seed=4)


@pytest.mark.parametrize("name", ["shuffle", "repeated", "predefined"])
def test_svc_all_scorers_general_splitters(engine, gap_binary, name):
    """Rows in neither set (shuffle, predefined) and overlapping test sets (repeated) through every fused scorer."""
    from sklearn.svm import SVC
    X, y = gap_binary
    cv = _general_cvs(y)[name]
    grid = {"C": [0.5, 5.0], "gamma": [0.05]}
    ref = _Fits(SVC(), _grid_cands(grid), X, y, list(cv.split(X, y)))
    _assert_svc_margin(ref, 2)
    for scoring in CLASSIFICATION_SCORERS:
        a = _search(SVC(), grid, X, y, cv, scoring)
        _assert_scores(a, ref, scoring, auc_delta=DELTA_SVC)


@pytest.mark.parametrize("name", ["kfold", "shuffle", "repeated", "predefined"])
def test_logreg_all_scorers(engine, gap_binary, name):
    """All nine classification scorers of binary LogisticRegression, on a partition and on the general splitters."""
    from sklearn.linear_model import LogisticRegression
    from sklearn.model_selection import StratifiedKFold
    X, y = gap_binary
    cv = StratifiedKFold(5) if name == "kfold" else _general_cvs(y)[name]
    grid = {"C": [0.01, 1.0]}
    ref = _Fits(LogisticRegression(), _grid_cands(grid), X, y, list(cv.split(X, y)))
    _assert_logreg_margin(ref)
    for scoring in CLASSIFICATION_SCORERS:
        a = _search(LogisticRegression(), grid, X, y, cv, scoring)
        _assert_scores(a, ref, scoring, auc_delta=DELTA_LOGREG)


@pytest.mark.parametrize("labels", [(0, 1), (-1, 1), (1, 2)])
@pytest.mark.parametrize("family", ["svc", "logreg"])
def test_label_encodings(engine, gap_binary, family, labels):
    """pos_label=1 is scikit-learn's positive class for f1 / precision / recall whatever the other label is: with {1, 2}
    it is the FIRST class.  roc_auc takes the greater label as positive."""
    from sklearn.linear_model import LogisticRegression
    from sklearn.model_selection import StratifiedKFold
    from sklearn.svm import SVC
    X, y01 = gap_binary
    y = np.where(y01 == 1, labels[1], labels[0])
    est, grid = (SVC(), {"C": [0.5, 5.0], "gamma": [0.05]}) if family == "svc" else (LogisticRegression(), {"C": [0.01, 1.0]})
    cv = StratifiedKFold(4)
    ref = _Fits(est, _grid_cands(grid), X, y, list(cv.split(X, y)))
    if family == "svc":
        _assert_svc_margin(ref, 2)
    else:
        _assert_logreg_margin(ref)
    for scoring in ("f1", "precision", "recall", "roc_auc"):
        a = _search(est, grid, X, y, cv, scoring)
        _assert_scores(a, ref, scoring, auc_delta=DELTA_SVC if family == "svc" else DELTA_LOGREG)


@pytest.mark.parametrize("family", ["svc", "logreg"])
def test_labels_without_pos_label_raise(engine, gap_binary, family):
    from sklearn.linear_model import LogisticRegression
    from sklearn.model_selection import GridSearchCV as SkGrid
    from sklearn.svm import SVC
    from spark_sklearn_b200 import GridSearchCV
    X, y01 = gap_binary
    y = np.where(y01 == 1, 5, 2)
    est = SVC() if family == "svc" else LogisticRegression()
    with pytest.raises(ValueError):
        GridSearchCV(None, est, {"C": [1.0]}, cv=3, scoring="f1").fit(X, y)
    with warnings.catch_warnings(), pytest.raises(ValueError):
        warnings.simplefilter("ignore")
        SkGrid(est, {"C": [1.0]}, cv=3, scoring="f1", error_score="raise").fit(X, y)


@pytest.mark.parametrize("family", ["svc", "logreg"])
def test_roc_auc_exact_ties(engine, gap_binary, family):
    """Duplicated rows with opposite labels in the same test set: equal scores on both sides, each pair counts 1/2."""
    from sklearn.linear_model import LogisticRegression
    from sklearn.model_selection import PredefinedSplit
    from sklearn.svm import SVC
    X0, y0 = gap_binary
    fold0 = np.arange(len(y0)) % 4
    dup = np.arange(0, len(y0), 7)
    X = np.concatenate([X0, X0[dup]])
    y = np.concatenate([y0, 1 - y0[dup]])
    cv = PredefinedSplit(np.concatenate([fold0, fold0[dup]]))
    est, grid, delta = ((SVC(), {"C": [0.5, 5.0], "gamma": [0.05]}, DELTA_SVC) if family == "svc"
                        else (LogisticRegression(), {"C": [0.01, 1.0]}, DELTA_LOGREG))
    ref = _Fits(est, _grid_cands(grid), X, y, list(cv.split(X, y)))
    ties = 0
    for (ci, k), s in ref.dec.items():
        te = ref.splits[k][1]
        sp, sn = s[te][y[te] == 1], s[te][y[te] == 0]
        ties += np.count_nonzero(sp[:, None] == sn[None, :])
    assert ties >= len(dup) * len(ref.cands)                      # the duplicates tie (at least) with each other
    a = _search(est, grid, X, y, cv, "roc_auc")
    _assert_scores(a, ref, "roc_auc", auc_delta=delta)


@pytest.mark.parametrize("family", ["svc", "logreg"])
def test_roc_auc_single_class_test_set(engine, gap_binary, family):
    """A test set with one class: roc_auc is undefined there; error_score=nan fills that split only, its train score
    stays finite, and the candidates still rank (NaN means last)."""
    from sklearn.linear_model import LogisticRegression
    from sklearn.model_selection import GridSearchCV as SkGrid, PredefinedSplit
    from sklearn.svm import SVC
    X, y = gap_binary
    fold = np.arange(len(y)) % 3
    fold[(y == 1) & (fold == 0)] = 1                               # test set 0 holds class 0 only
    cv = PredefinedSplit(fold)
    est, grid = (SVC(), {"C": [0.5, 5.0], "gamma": [0.05]}) if family == "svc" else (LogisticRegression(), {"C": [0.01, 1.0]})
    a = _search(est, grid, X, y, cv, "roc_auc", error_score=np.nan)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        b = SkGrid(est, grid, cv=cv, scoring="roc_auc", error_score=np.nan, return_train_score=True).fit(X, y)
    assert np.isnan(a.cv_results_["split0_test_score"]).all() and np.isnan(b.cv_results_["split0_test_score"]).all()
    assert np.isfinite(a.cv_results_["split0_train_score"]).all()
    tol = 1e-12 if family == "svc" else 2e-3
    for key in ("split0_train_score", "split1_test_score", "split2_test_score", "split1_train_score"):
        np.testing.assert_allclose(a.cv_results_[key], b.cv_results_[key], rtol=0, atol=tol, err_msg=key)
    np.testing.assert_array_equal(a.cv_results_["rank_test_score"], b.cv_results_["rank_test_score"])


@pytest.mark.parametrize("k", [5, 64])
def test_multinomial_logreg_scorers(engine, k):
    """Multinomial LogisticRegression up to the 64-class limit on well-separated blobs (5 % of labels flipped).  Small C:
    the fit converges in few iterations, so scikit-learn's and the float32-faithful logits stay close (DELTA_LOGREG_MULTI)."""
    from sklearn.linear_model import LogisticRegression
    from sklearn.model_selection import StratifiedKFold
    X, y = _blobs([40 + (i * 11) % 30 for i in range(k)], k, 12, seed=6, std=1.0, box=10.0)
    rng = np.random.RandomState(6)
    f = rng.rand(len(y)) < 0.05
    y = y.copy()
    y[f] = rng.randint(0, k, f.sum())
    cv = StratifiedKFold(4)
    grid = {"C": [0.002, 0.01]}
    ref = _Fits(LogisticRegression(), _grid_cands(grid), X, y, list(cv.split(X, y)))
    _assert_logreg_margin(ref, k)
    for scoring in MULTICLASS_SCORERS:
        a = _search(LogisticRegression(), grid, X, y, cv, scoring)
        _assert_scores(a, ref, scoring)


def test_logreg_65_classes_raises(engine):
    from sklearn.linear_model import LogisticRegression
    from spark_sklearn_b200 import GridSearchCV
    X, y = _blobs([10] * 65, 65, 8, seed=6)
    gs = GridSearchCV(None, LogisticRegression(), {"C": [1.0]}, cv=3)
    with pytest.raises(NotImplementedError, match="64 classes"):
        gs.fit(X, y)


# ------------------------------------------------------------------ 3. regression scorers ---------
def _regression(n=1200, d=20, seed=7):
    from sklearn.datasets import make_regression
    X, y = make_regression(n_samples=n, n_features=d, n_informative=12, noise=5.0, random_state=seed)
    return X.astype(np.float32), y.astype(np.float32)


def _assert_regression(a, b, scoring, n_splits, y):
    for k in range(n_splits):
        for part in ("test", "train"):
            key = "split%d_%s_score" % (k, part)
            # R^2: the per-split bar of test_gpu_enet.py (both solvers stop on the same duality gap).  MSE comes from Gram
            # statistics whose error is a fraction of the TOTAL sum of squares, not of the residual: the same bar in MSE units,
            # 5e-5 * var(y) (test_gpu_enet.py); RMSE is compared squared.
            ga, gb = a.cv_results_[key], b.cv_results_[key]
            if scoring == "r2":
                np.testing.assert_allclose(ga, gb, rtol=0, atol=5e-5, err_msg=key)
            else:
                if scoring == "neg_root_mean_squared_error":
                    ga, gb = -ga * ga, -gb * gb
                np.testing.assert_allclose(ga, gb, rtol=0, atol=5e-5 * np.var(y), err_msg=key)


@pytest.mark.parametrize("scoring", ["r2", "neg_mean_squared_error", "neg_root_mean_squared_error"])
@pytest.mark.parametrize("splitter", ["kfold", "shuffle"])
@pytest.mark.parametrize("family", ["lasso", "elasticnet"])
def test_enet_regression_scorers(engine, family, splitter, scoring):
    from sklearn.linear_model import ElasticNet, Lasso
    from sklearn.model_selection import GridSearchCV as SkGrid, KFold, ShuffleSplit
    X, y = _regression()
    cv = KFold(4) if splitter == "kfold" else ShuffleSplit(3, test_size=0.25, train_size=0.6, random_state=3)
    est, grid = ((Lasso(), {"alpha": [0.05, 1.0, 10.0]}) if family == "lasso"
                 else (ElasticNet(), {"alpha": [0.05, 1.0], "l1_ratio": [0.2, 0.8]}))
    a = _search(est, grid, X, y, cv, None if scoring == "r2" else scoring)
    b = SkGrid(est, grid, cv=cv, scoring=scoring, return_train_score=True).fit(X, y)
    _assert_regression(a, b, scoring, b.n_splits_, y)


@pytest.mark.parametrize("scoring", ["r2", "neg_mean_squared_error"])
@pytest.mark.parametrize("family", ["ridge", "lasso"])
def test_constant_target_test_fold(engine, family, scoring):
    """A test fold whose targets are all equal: scikit-learn's r2_score is 0.0 there (the total sum of squares is 0;
    force_finite), and so is the search's, instead of 1 - res / (rounding noise)."""
    from sklearn.linear_model import Lasso, Ridge
    from sklearn.model_selection import GridSearchCV as SkGrid, PredefinedSplit
    X, y = _regression()
    fold = np.arange(len(y)) % 4
    # float64 targets: scikit-learn's r2_score on a float32 constant set divides by the rounding error of its float32
    # mean (-2e19 here), on float64 by an exact 0
    y = y.astype(np.float64)
    y[fold == 0] = float(np.float32(np.median(y)))
    cv = PredefinedSplit(fold)
    est, grid = (Ridge(), {"alpha": [0.1, 10.0]}) if family == "ridge" else (Lasso(), {"alpha": [0.05, 1.0]})
    a = _search(est, grid, X, y, cv, None if scoring == "r2" else scoring)
    b = SkGrid(est, grid, cv=cv, scoring=scoring, return_train_score=True).fit(X, y)
    if scoring == "r2":
        assert (b.cv_results_["split0_test_score"] == 0.0).all()
        assert (a.cv_results_["split0_test_score"] == 0.0).all(), a.cv_results_["split0_test_score"]
        for key in ("split1_test_score", "split0_train_score", "split1_train_score"):
            np.testing.assert_allclose(a.cv_results_[key], b.cv_results_[key], rtol=0, atol=5e-5, err_msg=key)
    else:
        _assert_regression(a, b, scoring, 4, y)
