"""Search driver: the B200 counterpart of ``SparkBaseSearchCV._fit``
(reference python/spark_sklearn/base_search.py:21-175).

Same steps, same order, same result layout as the reference -- ``check_cv`` / reseed
(:34-41), ``check_scoring`` (:43), the "Fitting K folds..." message (:48-52), the candidate-major
fold-minor task list (:56-61), ``_store`` aggregation with the ``iid`` test-size weighting
(:100-137), ``rankdata(-mean, 'min')`` (:123-125), masked ``param_*`` arrays (:145-156), refit
(:165-174) -- except that the Spark fan-out ``parallelize(...).map(fun).collect()`` (:62-98) is ONE
call into libb200gs.so that evaluates the whole task list on the GPU (``estimators.py``).
With ``torch.distributed`` initialised (one process per GPU) the candidates are dealt (by predicted cost) over the
ranks and the per-candidate score blocks are exchanged with a single all-gather -- the
counterpart of ``collect()``.
"""
import time
from collections import defaultdict
from functools import partial
from random import randint

import numpy as np
from numpy.ma import MaskedArray
from scipy.stats import rankdata
from sklearn.base import clone, is_classifier
from sklearn.metrics import check_scoring
from sklearn.model_selection import check_cv
from sklearn.model_selection._search import BaseSearchCV
from sklearn.utils.validation import indexable

from . import estimators as _est
from . import dist as _dist


class B200BaseSearchCV(BaseSearchCV):
    """Drop-in for ``spark_sklearn.base_search.SparkBaseSearchCV`` (reference base_search.py:21-29)."""

    def __init__(self, estimator, scoring=None, fit_params=None, n_jobs=1, iid=True, refit=True, cv=None,
                 verbose=0, pre_dispatch='2*n_jobs', error_score='raise', return_train_score=True):
        self.estimator = estimator
        self.scoring = scoring
        self.fit_params = fit_params
        self.n_jobs = n_jobs            # accepted and ignored, as in the reference (grid_search.py:46-50)
        self.iid = iid
        self.refit = refit
        self.cv = cv
        self.verbose = verbose
        self.pre_dispatch = pre_dispatch
        self.error_score = error_score
        self.return_train_score = return_train_score

    # sklearn >= 1.6 validates constructor params of BaseSearchCV subclasses through
    # _parameter_constraints when its own fit() runs; this class has its own _fit.
    def _run_search(self, evaluate_candidates):  # pragma: no cover - abstract in sklearn, unused here
        raise NotImplementedError

    def _fit(self, X, y, groups, parameter_iterable):
        estimator = self.estimator
        cv = check_cv(self.cv, y, classifier=is_classifier(estimator))
        if hasattr(cv, 'random_state'):                       # reference base_search.py:39-41
            if not cv.random_state:
                cv.random_state = randint(1000, 9999)
        self.scorer_ = check_scoring(self.estimator, scoring=self.scoring)
        self.multimetric_ = False

        X, y, groups = indexable(X, y, groups)
        splits = list(cv.split(X, y, groups))
        n_splits = len(splits)
        candidate_params = [dict(p) for p in parameter_iterable]
        rank, world = _dist.rank_world()
        if world > 1:                                         # one candidate list and one set of folds for all ranks: rank 0's
            candidate_params, splits = _dist.broadcast_plan((candidate_params, splits))
            n_splits = len(splits)
        n_param_candidates = len(candidate_params)
        if self.verbose > 0:                                  # reference base_search.py:48-52
            print("Fitting {0} folds for each of {1} candidates, totalling"
                  " {2} fits".format(n_splits, n_param_candidates, n_param_candidates * n_splits))

        adapter = _est.adapter_for(estimator)                 # raises for estimators without a CUDA path
        if self.scoring is not None and (not isinstance(self.scoring, str) or self.scoring not in getattr(adapter, "scorers", {})):
            raise NotImplementedError(
                "scoring=%r has no fused CUDA scorer for %s (available: %s); callables and multi-metric scoring would need "
                "the fitted estimators on the host and there is no CPU fallback"
                % (self.scoring, type(estimator).__name__, sorted(k for k in getattr(adapter, "scorers", {}) if k)))
        X_arr = X.toarray() if hasattr(X, "toarray") else np.asarray(X)     # scipy.sparse input: the engine is dense
        y_arr = None if y is None else np.asarray(y)
        fold_id = _est.Folds(splits, len(X_arr))               # fold ids for partition splitters, split masks otherwise

        # ---- the fan-out: every (candidate, fold) task in one engine call per GPU ----
        devices = _dist.local_devices() if (world == 1 and getattr(adapter, "multi_device", False)) else [None]
        devices = devices[:max(1, n_param_candidates)]
        if len(devices) > 1:
            # the in-process scheduler: ONE fit() drives every visible GPU -- a handle and a host thread per device (ctypes
            # releases the GIL for the whole gs_* call), the dataset uploaded once to each, candidates dealt by predicted cost,
            # score blocks merged on the host.  The counterpart of sc.parallelize(tasks).map(fun).collect() on one node.
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(len(devices)) as pool:
                plans = list(pool.map(lambda d: adapter.plan(clone(estimator), candidate_params, X_arr, y_arr, fold_id, n_splits,
                                                             device=d), devices))
                for p in plans:
                    if self.scoring is not None or hasattr(p, "set_scoring"):
                        p.set_scoring(self.scoring)           # raises for scorers without a fused CUDA path
                    if self.fit_params or hasattr(p, "set_fit_params"):
                        p.set_fit_params(self.fit_params)     # sample_weight; raises for anything without a CUDA path
                parts = _dist.assign_for_plan(plans[0], n_param_candidates, len(devices))
                locs = list(pool.map(lambda i: plans[i].evaluate(parts[i], return_train=self.return_train_score,
                                                                 error_score=self.error_score) if parts[i] else None,
                                     range(len(devices))))
            out = _dist.merge_candidates(locs, parts, n_param_candidates, n_splits)
            plan = plans[0]
            self.device_profile_ = _dist.merge_profiles([p.profile() for p in plans])
            self.devices_ = list(devices)
            for p in plans[1:]:
                p.close()
        else:
            plan = adapter.plan(clone(estimator), candidate_params, X_arr, y_arr, fold_id, n_splits)
            if self.scoring is not None or hasattr(plan, "set_scoring"):
                plan.set_scoring(self.scoring)                # raises for scorers without a fused CUDA path
            if self.fit_params or hasattr(plan, "set_fit_params"):
                plan.set_fit_params(self.fit_params)          # sample_weight; raises for anything without a CUDA path
            # candidates dealt to the GPUs by predicted cost (the reference leaves the placement of its tasks to Spark)
            parts = _dist.assign_for_plan(plan, n_param_candidates, world)
            my = parts[rank]
            local = plan.evaluate(my, return_train=self.return_train_score, error_score=self.error_score)
            out = _dist.allgather_candidates(local, my, n_param_candidates, n_splits, world, parts,
                                             device=getattr(getattr(plan, "engine", None), "device", None))
            self.device_profile_ = plan.profile()
            self.devices_ = [getattr(getattr(plan, "engine", None), "device", None)]
        test_scores, train_scores = out["test"], out["train"]
        fit_time, score_time = out["fit_time"], out["score_time"]

        test_sample_counts = np.array([len(te) for _, te in splits], dtype=int)
        results = dict()

        def _store(key_name, array, weights=None, splits=False, rank=False):
            """reference base_search.py:100-125"""
            array = np.array(array, dtype=np.float64).reshape(n_param_candidates, n_splits)
            if splits:
                for split_i in range(n_splits):
                    results["split%d_%s" % (split_i, key_name)] = array[:, split_i]
            array_means = np.average(array, axis=1, weights=weights)
            results['mean_%s' % key_name] = array_means
            array_stds = np.sqrt(np.average((array - array_means[:, np.newaxis]) ** 2, axis=1, weights=weights))
            results['std_%s' % key_name] = array_stds
            if rank:
                # a NaN mean (a split scored error_score=nan) ranks last, as in scikit-learn; all NaN: all rank 1
                if np.isnan(array_means).all():
                    ranked = np.ones_like(array_means)
                else:
                    ranked = rankdata(-np.nan_to_num(array_means, nan=np.nanmin(array_means) - 1), method='min')
                results["rank_%s" % key_name] = np.asarray(ranked, dtype=np.int32)

        _store('test_score', test_scores, splits=True, rank=True,
               weights=test_sample_counts if self.iid else None)
        if self.return_train_score:
            _store('train_score', train_scores, splits=True)
        _store('fit_time', fit_time)
        _store('score_time', score_time)

        best_index = np.flatnonzero(results["rank_test_score"] == 1)[0]
        best_parameters = candidate_params[best_index]

        param_results = defaultdict(partial(MaskedArray, np.empty(n_param_candidates,), mask=True, dtype=object))
        for cand_i, params in enumerate(candidate_params):
            for name, value in params.items():
                param_results["param_%s" % name][cand_i] = value
        results.update(param_results)
        results['params'] = candidate_params

        self.cv_results_ = results
        self.best_index_ = best_index
        self.n_splits_ = n_splits
        self.best_params_ = best_parameters
        self.best_score_ = results["mean_test_score"][best_index]

        if self.refit:                                         # reference base_search.py:165-174
            t0 = time.time()
            self.best_estimator_ = plan.refit(best_parameters)
            self.refit_time_ = time.time() - t0
        plan.close()
        return self
