"""Cross-validation and grid search whose SMO fits share Gram matrices on the GPU.

``sklearn.model_selection.GridSearchCV(SVC(optimizer='smo', ...), {'C': [...]}, cv=5)`` clones the estimator for every
(candidate, fold) pair and fits the clones one after the other: every fit uploads X, builds its own Gram matrix and
runs one SMO solve that leaves most of the GPU idle.  The drop-ins below keep sklearn's contract and fit the same
clones through ``ml.multiclass.fit_shared_gram`` instead: the problems whose kernel resolves to the same spec share ONE
matrix, built on the union of their training rows, and run side by side in one SMO batch (``svmb200_smo_run_batch``).

A training fold T is the problem on the whole matrix with every variable outside T held at 0
(``svmb200_smo_create_subset``): such a variable is never selected, ties go to the larger index and the map from T's
own indices to the matrix's is monotone, and K1 computes every element of the matrix from its two samples alone.  So
every clone ends bit for bit where ``clone(est).set_params(**p).fit(X[T], y[T])`` ends on the same GPU, and
``cv_results_``, ``best_index_``, ``best_params_``, ``best_score_`` and ``best_estimator_`` equal sklearn's.

Timing keys: a problem's ``fit_time`` is the wall clock of its group (upload, Gram matrix, batch, finishing every
clone) divided by the problems in the group; ``score_time`` is measured per problem, as sklearn does.

Everything else goes through sklearn's own implementation, unchanged: fit parameters or sample weights, metadata
routing, callbacks, ``verbose``, estimators other than this package's ``optimizer='smo'`` ``SVC`` / ``SVR``, a
training fold that does not hold exactly two classes (sklearn's errors and ``error_score``), a context that would
shard the matrix over several GPUs, and a candidate whose fit raises a ValueError, TypeError or NotImplementedError.
"""
import time
from collections import defaultdict
from itertools import product

import numpy as np
from sklearn import model_selection as _skms
from sklearn.base import clone, is_classifier
from sklearn.metrics import check_scoring
from sklearn.metrics._scorer import _MultimetricScorer
from sklearn.model_selection import ParameterGrid, check_cv
from sklearn.model_selection._validation import (_aggregate_score_dicts, _normalize_score_results, _safe_split,
                                                 _score)
from sklearn.utils import _safe_indexing, indexable
from sklearn.utils._metadata_requests import _routing_enabled
from sklearn.utils.validation import _num_samples

from .ml.multiclass import _smo_batch_capable, fit_shared_gram
from .ml.svm import SVC, SVR
from .runtime import would_shard

__all__ = ['GridSearchCV', 'cross_validate', 'cross_val_score']


def _fit_and_score_shared(estimator, X, y, candidates, splits, scorer, return_train_score, error_score,
                          return_estimator=False):
    """sklearn's ``_fit_and_score`` outputs for every (candidate, split) pair, candidate-major, with the fits shared
    through ``fit_shared_gram``; None when a problem is outside the shared path (the caller then runs sklearn's)."""
    if y is None or _routing_enabled() or not isinstance(estimator, (SVC, SVR)):
        return None
    if not all(_smo_batch_capable(clone(estimator).set_params(**clone(p or {}, safe=False))) for p in candidates):
        return None
    if any(would_shard(len(train)) for train, _ in splits):
        return None
    if is_classifier(estimator) and any(len(np.unique(_safe_indexing(y, train))) != 2 for train, _ in splits):
        return None
    problems = [(p, _safe_split(estimator, X, y, train)[1], train) for p, (train, _) in product(candidates, splits)]
    try:
        fitted = fit_shared_gram(estimator, X, problems)
    except (ValueError, TypeError, NotImplementedError):
        return None   # sklearn's implementation reports the failing fit its own way (error_score)
    out = []
    for est, (train, test) in zip(fitted, [s for _ in candidates for s in splits]):
        X_test, y_test = _safe_split(est, X, y, test, train)
        t0 = time.time()
        result = {'fit_error': None, 'test_scores': _score(est, X_test, y_test, scorer, {}, error_score)}
        score_time = time.time() - t0
        if return_train_score:
            X_train, y_train = _safe_split(est, X, y, train)
            result['train_scores'] = _score(est, X_train, y_train, scorer, {}, error_score)
        result.update(n_test_samples=_num_samples(X_test), fit_time=est.fit_times_['share_s'], score_time=score_time)
        if return_estimator:
            result['estimator'] = est
        out.append(result)
    return out


class GridSearchCV(_skms.GridSearchCV):
    """``sklearn.model_selection.GridSearchCV`` whose SMO fits share Gram matrices (module docstring).  The refit of
    the best candidate is an ordinary single fit."""

    def fit(self, X, y=None, **params):
        if params or self.verbose or getattr(self, '_skl_callbacks', None):
            return super().fit(X, y, **params)
        self._validate_params()
        scorers, refit_metric = self._get_scorers()
        Xi, yi = indexable(X, y)
        cv = check_cv(self.cv, yi, classifier=is_classifier(self.estimator))
        n_splits = cv.get_n_splits(Xi, yi)
        splits = list(cv.split(Xi, yi))
        if len(splits) != n_splits:
            raise ValueError(f'cv.split and cv.get_n_splits return inconsistent results. Expected {n_splits} splits, '
                             f'got {len(splits)}')
        candidates = list(ParameterGrid(self.param_grid))
        out = _fit_and_score_shared(self.estimator, Xi, yi, candidates, splits, scorers, self.return_train_score,
                                    self.error_score)
        if out is None:
            return super().fit(X, y)
        self._checked_cv_orig, self.n_splits_ = cv, n_splits
        # from here on, what sklearn's fit does with the outputs of its own fits
        results = self._format_results(candidates, n_splits, out, defaultdict(list))
        first_test_score = out[0]['test_scores']
        self.multimetric_ = isinstance(first_test_score, dict)
        if callable(self.scoring) and self.multimetric_:
            self._check_refit_for_multimetric(first_test_score)
            refit_metric = self.refit
        if self.refit or not self.multimetric_:
            self.best_index_ = self._select_best_index(self.refit, refit_metric, results)
            if not callable(self.refit):
                self.best_score_ = results[f'mean_test_{refit_metric}'][self.best_index_]
            self.best_params_ = results['params'][self.best_index_]
        if self.refit:
            self.best_estimator_ = clone(self.estimator).set_params(**clone(self.best_params_, safe=False))
            t0 = time.time()
            self.best_estimator_.fit(Xi, yi)
            self.refit_time_ = time.time() - t0
            if hasattr(self.best_estimator_, 'feature_names_in_'):
                self.feature_names_in_ = self.best_estimator_.feature_names_in_
        self.scorer_ = scorers._scorers if isinstance(scorers, _MultimetricScorer) else scorers
        self.cv_results_ = results
        return self


def cross_validate(estimator, X, y=None, *, groups=None, scoring=None, cv=None, n_jobs=None, verbose=0, params=None,
                   pre_dispatch='2*n_jobs', return_train_score=False, return_estimator=False, return_indices=False,
                   error_score=np.nan):
    """``sklearn.model_selection.cross_validate`` whose SMO fits share one Gram matrix (module docstring)."""
    sk_args = dict(groups=groups, scoring=scoring, cv=cv, n_jobs=n_jobs, verbose=verbose, params=params,
                   pre_dispatch=pre_dispatch, return_train_score=return_train_score,
                   return_estimator=return_estimator, return_indices=return_indices, error_score=error_score)
    if params or verbose:
        return _skms.cross_validate(estimator, X, y, **sk_args)
    Xi, yi = indexable(X, y)
    cvi = check_cv(cv, yi, classifier=is_classifier(estimator))
    scorers = check_scoring(estimator, scoring=scoring, raise_exc=(error_score == 'raise'))
    splits = list(cvi.split(Xi, yi, groups))
    out = _fit_and_score_shared(estimator, Xi, yi, [None], splits, scorers, return_train_score, error_score,
                                return_estimator)
    if out is None:
        return _skms.cross_validate(estimator, X, y, **sk_args)
    # sklearn's assembly of the returned dict
    results = _aggregate_score_dicts(out)
    ret = {'fit_time': results['fit_time'], 'score_time': results['score_time']}
    if return_estimator:
        ret['estimator'] = results['estimator']
    if return_indices:
        ret['indices'] = {}
        ret['indices']['train'], ret['indices']['test'] = zip(*splits)
    test_scores_dict = _normalize_score_results(results['test_scores'])
    if return_train_score:
        train_scores_dict = _normalize_score_results(results['train_scores'])
    for name in test_scores_dict:
        ret[f'test_{name}'] = test_scores_dict[name]
        if return_train_score:
            ret[f'train_{name}'] = train_scores_dict[name]
    return ret


def cross_val_score(estimator, X, y=None, *, groups=None, scoring=None, cv=None, n_jobs=None, verbose=0, params=None,
                    pre_dispatch='2*n_jobs', error_score=np.nan):
    """``sklearn.model_selection.cross_val_score`` on top of this module's ``cross_validate``."""
    scorer = check_scoring(estimator, scoring=scoring)
    cv_results = cross_validate(estimator=estimator, X=X, y=y, groups=groups, scoring={'score': scorer}, cv=cv,
                                n_jobs=n_jobs, verbose=verbose, params=params, pre_dispatch=pre_dispatch,
                                error_score=error_score)
    return cv_results['test_score']
