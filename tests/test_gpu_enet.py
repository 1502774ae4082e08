"""GPU parity tests for Lasso / ElasticNet (SURVEY.md 8f-2; the estimator of the reference's own search tests,
python/spark_sklearn/tests/test_search_2.py:69-119) through the C ABI: fold Grams + Gram-domain coordinate descent.

Checker: goldens made by scikit-learn 1.9.0, the numpy restatement of its coordinate descent (oracle.enet_cd), and
scikit-learn's GridSearchCV itself.  Floating point: both sides stop on the same duality-gap rule (tol * ||y||^2), so the
coefficients agree to the solver tolerance, not to the last bit; 5e-5 on per-split R^2 (BASELINE: 1e-4 on mean_test_score).
The sweep counts must agree except where a stopping test falls within rounding of its threshold."""
import warnings

import numpy as np
import pytest

from conftest import golden
from spark_sklearn_b200 import workloads as W

pytestmark = pytest.mark.gpu


def _setup(engine, key):
    from oracle import oracle as O
    w = W.make_workload(key)
    fold_id, ns = O.folds_from_cv(w["cv"], w["X"], w["y"], False)
    engine.set_data(w["X"], fold_id, ns, y_target=w["y"])
    return w, fold_id, ns


@pytest.mark.parametrize("key", ["lasso_small", "enet_small"])
def test_enet_vs_golden_and_oracle(engine, key):
    from oracle import oracle as O
    w, fold_id, ns = _setup(engine, key)
    g = golden(key)
    cands = W.candidates(w)
    r = engine.enet([c["alpha"] for c in cands], [c.get("l1_ratio", 1.0) for c in cands])
    assert np.abs(r["test"] - g["test_scores"]).max() <= 5e-5
    assert np.abs(r["train"] - g["train_scores"]).max() <= 5e-5
    assert np.abs(r["test"].mean(1) - g["test_scores"].mean(1)).max() <= 2e-5
    n_iter = g["diag"][:, :, 0].astype(int)
    assert (r["n_iter"] == n_iter).mean() >= 0.9 and np.abs(r["n_iter"] - n_iter).max() <= 2, (r["n_iter"], n_iter)
    te, tr, it = O.cv_scores_enet(w["X"], w["y"], fold_id, ns, cands[::5])
    assert np.abs(r["test"][::5] - te).max() <= 5e-5 and np.abs(r["train"][::5] - tr).max() <= 5e-5


def test_enet_no_intercept_ragged_folds_and_corners(engine):
    """d not a multiple of 32, unequal folds, no intercept; alpha large enough for w = 0 (n_iter 0), alpha = 0 with an
    L2 term only (duality gap formulation B), a duplicated and an all-zero column (screened out)."""
    from oracle import oracle as O
    rng = np.random.RandomState(3)
    n, d = 777, 45
    X = (rng.randn(n, d) + 1.0).astype(np.float32)
    X[:, 7] = X[:, 3]
    X[:, 11] = 0.0
    y = (X[:, :10] @ rng.randn(10) + 0.5 * rng.randn(n) + 2).astype(np.float32)
    fold_id, ns = O.folds_from_cv(7, X, y, False)
    engine.set_data(X, fold_id, ns, y_target=y)
    cands = [dict(alpha=a, l1_ratio=l) for a, l in ((1e-3, 1.0), (0.05, 1.0), (0.3, 0.5), (0.2, 0.0), (1e4, 1.0), (2.0, 0.9))]
    for fi in (True, False):
        r = engine.enet([c["alpha"] for c in cands], [c["l1_ratio"] for c in cands], fit_intercept=fi)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            te, tr, it = O.cv_scores_enet(X, y, fold_id, ns, cands, fit_intercept=fi)
        assert np.abs(r["test"] - te).max() <= 5e-5, (fi, np.abs(r["test"] - te).max())
        assert np.abs(r["train"] - tr).max() <= 5e-5, (fi, np.abs(r["train"] - tr).max())
        assert np.abs(r["n_iter"] - it).max() <= 2, (fi, r["n_iter"], it)
        if fi:
            assert (r["n_iter"][4] == 0).all()             # w = 0 is optimal: scikit-learn returns before the first sweep


def test_lasso_python_api_refit_and_reference_style_pipeline(engine):
    """GridSearchCV(Lasso) against scikit-learn's GridSearchCV; then the reference's own test shape: a one-step Pipeline
    searched through 'lasso__alpha' on a scipy.sparse X with a column-vector y (reference tests/test_search_2.py:69-80)."""
    import scipy.sparse
    from sklearn.linear_model import Lasso
    from sklearn.model_selection import GridSearchCV as SkGrid
    from sklearn.pipeline import Pipeline
    from spark_sklearn_b200 import GridSearchCV, RandomizedSearchCV
    w = W.make_workload("lasso_small")
    X, y = w["X"], w["y"]
    grid = {"alpha": [0.01, 0.3, 3.0, 30.0], "fit_intercept": [True, False]}
    a = GridSearchCV(None, Lasso(), grid, cv=4, iid=False).fit(X, y)
    b = SkGrid(Lasso(), grid, cv=4, return_train_score=True).fit(X, y)
    for key in ("mean_test_score", "mean_train_score", "std_test_score"):
        np.testing.assert_allclose(a.cv_results_[key], b.cv_results_[key], atol=2e-5, err_msg=key)
    assert a.best_params_ == b.best_params_
    ea, eb = a.best_estimator_, b.best_estimator_
    np.testing.assert_allclose(ea.coef_, eb.coef_, atol=2e-4 * np.abs(eb.coef_).max())
    assert ((ea.coef_ != 0) == (eb.coef_ != 0)).mean() >= 0.95
    np.testing.assert_allclose(ea.intercept_, eb.intercept_, atol=1e-3)
    assert abs(ea.n_iter_ - eb.n_iter_) <= 1
    np.testing.assert_allclose(a.predict(X), b.predict(X), atol=2e-3 * np.abs(y).max())

    Xs = scipy.sparse.csr_matrix(np.array([[float(i), i + 1.0] for i in range(100)]))
    ys = np.arange(100, dtype=float).reshape(100, 1)
    params = {"lasso__alpha": (0.001, 0.005, 0.01)}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gs = GridSearchCV(None, Pipeline([("lasso", Lasso())]), params).fit(Xs, ys)
        ref = SkGrid(Pipeline([("lasso", Lasso())]), params, cv=3).fit(Xs, ys)
    assert len(gs.cv_results_["params"]) == 3                     # the reference test's own assertion
    np.testing.assert_allclose(gs.cv_results_["mean_test_score"], ref.cv_results_["mean_test_score"], rtol=2e-4, atol=2e-4)
    assert gs.best_estimator_.named_steps["lasso"].coef_.shape == (1, 2) or gs.best_estimator_.named_steps["lasso"].coef_.shape == (2,)
    np.testing.assert_allclose(np.ravel(gs.predict(Xs.toarray())), np.ravel(ref.predict(Xs)), rtol=1e-3, atol=1e-2)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        rs = RandomizedSearchCV(None, Pipeline([("lasso", Lasso(max_iter=1))]), {"lasso__alpha": np.linspace(0.001, 0.01, 1000)},
                                n_iter=10).fit(Xs, ys)            # reference tests/test_search_2.py:82-93
    assert len(rs.cv_results_["params"]) == 10


def test_elasticnet_general_splitter_and_mse_scoring(engine):
    from sklearn.linear_model import ElasticNet
    from sklearn.model_selection import GridSearchCV as SkGrid, ShuffleSplit
    from spark_sklearn_b200 import GridSearchCV
    w = W.make_workload("enet_small")
    X, y = w["X"], w["y"]
    cv = ShuffleSplit(3, test_size=0.25, train_size=0.6, random_state=1)    # non-zero: the search redraws a falsy seed
    grid = {"alpha": [0.05, 1.0], "l1_ratio": [0.3, 0.9]}
    a = GridSearchCV(None, ElasticNet(), grid, cv=cv, iid=False, scoring="neg_mean_squared_error").fit(X, y)
    b = SkGrid(ElasticNet(), grid, cv=cv, return_train_score=True, scoring="neg_mean_squared_error").fit(X, y)
    for k in range(3):
        for part in ("test", "train"):
            key = "split%d_%s_score" % (k, part)
            # the R^2 bar (5e-5) expressed in MSE units: both solvers stop on a duality gap of 1e-4 * ||y||^2
            np.testing.assert_allclose(a.cv_results_[key], b.cv_results_[key], rtol=0, atol=5e-5 * np.var(y), err_msg=key)
    assert a.best_params_ == b.best_params_


def test_lasso_1024_features_vs_golden(engine):
    """Config 5's data (20000 x 1024, cv=10) with Lasso: 320 fits, eight registers-tiles of q per lane."""
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lasso_1024.npz")
    if not os.path.exists(path):
        pytest.skip("tests/golden/lasso_1024.npz not generated")
    w, fold_id, ns = _setup(engine, "lasso_1024")
    g = golden("lasso_1024")
    cands = W.candidates(w)
    r = engine.enet([c["alpha"] for c in cands], 1.0)
    assert np.abs(r["test"] - g["test_scores"]).max() <= 5e-5
    assert np.abs(r["test"].mean(1) - g["test_scores"].mean(1)).max() <= 2e-5
    n_iter = g["diag"][:, :, 0].astype(int)
    assert np.abs(r["n_iter"] - n_iter).max() <= 2


def _reference_tasks(est, grid, cv, X, y, sw, classifier=False):
    """The reference's own task (base_search.py:74-88 with scikit-learn <0.20's _fit_and_score): fit_params are sliced by the
    training rows and given to fit(); the scorer gets no weights.  (scikit-learn >= 1.4's GridSearchCV.fit(sample_weight=)
    also weights the scorer, so it is not the checker here.)  -> mean test / train score per candidate, fitted best"""
    from sklearn.base import clone
    from sklearn.model_selection import ParameterGrid, check_cv
    splits = list(check_cv(cv, y, classifier=classifier).split(X, y))
    cands = list(ParameterGrid(grid))
    te = np.zeros((len(cands), len(splits)))
    tr = np.zeros_like(te)
    for ci, p in enumerate(cands):
        for k, (a, b) in enumerate(splits):
            m = clone(est).set_params(**p).fit(X[a], y[a], sample_weight=sw[a])
            te[ci, k], tr[ci, k] = m.score(X[b], y[b]), m.score(X[a], y[a])
    best = int(np.argmax(te.mean(1)))
    return te.mean(1), tr.mean(1), cands[best], clone(est).set_params(**cands[best]).fit(X, y, sample_weight=sw)


def test_sample_weight_fit_params_linear_models(engine):
    """fit_params={'sample_weight': w} (reference base_search.py:69,83-87): the fit is weighted, the scores are not."""
    from sklearn.linear_model import ElasticNet, Lasso, Ridge
    from sklearn.model_selection import ShuffleSplit
    from spark_sklearn_b200 import GridSearchCV
    w = W.make_workload("lasso_small")
    X, y = w["X"], w["y"]
    rng = np.random.RandomState(5)
    sw = rng.gamma(1.0, 1.0, len(y))
    sw[rng.rand(len(y)) < 0.1] = 0.0                                  # some rows switched off
    for est, grid, cv in ((Ridge(), {"alpha": [1e-2, 10.0, 1e3]}, 4),
                          (Lasso(), {"alpha": [0.05, 2.0, 40.0]}, 4),
                          (ElasticNet(), {"alpha": [0.1, 3.0], "l1_ratio": [0.3, 0.8]}, ShuffleSplit(3, test_size=0.25, random_state=1))):
        a = GridSearchCV(None, est, grid, cv=cv, iid=False, fit_params={"sample_weight": sw}).fit(X, y)
        te, tr, best, fitted = _reference_tasks(est, grid, cv, X, y, sw)
        u = GridSearchCV(None, est, grid, cv=cv, iid=False).fit(X, y)
        name = type(est).__name__
        np.testing.assert_allclose(a.cv_results_["mean_test_score"], te, atol=5e-5, err_msg=name)
        np.testing.assert_allclose(a.cv_results_["mean_train_score"], tr, atol=5e-5, err_msg=name)
        assert np.abs(a.cv_results_["mean_train_score"] - u.cv_results_["mean_train_score"]).max() > 1e-5, name   # the weights matter
        assert a.best_params_ == best
        np.testing.assert_allclose(a.best_estimator_.coef_, fitted.coef_, atol=3e-4 * np.abs(fitted.coef_).max())
        np.testing.assert_allclose(a.best_estimator_.intercept_, fitted.intercept_, atol=2e-3)
    from sklearn.svm import SVC
    wc = W.make_workload("c2_small")
    with pytest.raises(NotImplementedError):
        GridSearchCV(None, SVC(), {"C": [1.0]}, cv=3, fit_params={"sample_weight": np.ones(len(wc["y"]))}).fit(wc["X"], wc["y"])
    with pytest.raises(NotImplementedError):
        GridSearchCV(None, Ridge(), {"alpha": [1.0]}, cv=3, fit_params={"check_input": False}).fit(X, y)
