"""Shared checks of cross-validation and grid search on shared Gram matrices (``svmb200_smo_create_subset``,
``ml/multiclass.py::fit_shared_gram`` with training rows, ``optiml_b200/model_selection.py``): the CPU suite runs them
on the host emulation, the GPU suite on the B200."""
import warnings
from unittest import mock

import numpy as np
from sklearn.base import clone
from sklearn.exceptions import ConvergenceWarning

import smo_batch_checks as SB


def kernels():
    from optiml_b200.ml.svm.kernels import GaussianKernel, LaplacianKernel, LinearKernel, PolyKernel, SigmoidKernel
    return {'linear': LinearKernel(), 'poly': PolyKernel(degree=3, gamma=0.3, coef0=1.0),
            'gaussian': GaussianKernel(gamma=0.2), 'laplacian': LaplacianKernel(gamma=0.1),
            'sigmoid': SigmoidKernel(gamma=0.05, coef0=0.5)}


def ragged_rows(n, k, seed=0):
    """k sorted training sets of uneven sizes: each leaves out a random block and a random scatter of rows"""
    rng = np.random.default_rng(seed)
    out = []
    for f in range(k):
        keep = rng.random(n) > 0.1 + 0.05 * f
        lo = rng.integers(0, n // 2)
        keep[lo:lo + rng.integers(1, n // 4)] = False
        out.append(np.flatnonzero(keep))
    return out


def gram_of(est, X, layout):
    """K1's unsigned M (bias 0) of X, on the host"""
    H = est._build_hessian(X, None, layout, None, 0.0)
    est._train_X_device[0].release()
    try:
        return H.shard_to_host()
    finally:
        H.release()


def check_sub_gram(kernel, X, rows, layout='plain'):
    """M of X restricted to `rows` equals M of X[rows], bit for bit (signed zeros and NaN payloads included)"""
    est = SB.svc(kernel)
    full = gram_of(est, X, layout)
    for r in rows:
        part = gram_of(est, X[r], layout)
        assert np.array_equal(full[np.ix_(r, r)].view(np.int64), part.view(np.int64))


def fit_fold(est, X, y, rows):
    """the clone path: one fit on the training rows alone; returns the clone and its ConvergenceWarnings"""
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        own = clone(est).fit(X[rows], y[rows])
    return own, sum(issubclass(x.category, ConvergenceWarning) for x in w)


def check_folds_equal_own_fits(est, X, y, rows, params=None):
    """fit_shared_gram on (params, y[T], T) problems against one clone fit per problem, bit for bit; returns both"""
    from optiml_b200.ml.multiclass import fit_shared_gram
    params = params or [{}]
    problems = [(p, y[r], r) for p in params for r in rows]
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        ours = fit_shared_gram(est, X, problems)
    conv = sum(issubclass(x.category, ConvergenceWarning) for x in w)
    theirs, conv_theirs = [], 0
    for p, t, r in problems:
        own, c = fit_fold(clone(est).set_params(**p), X, y, r)
        theirs.append(own)
        conv_theirs += c
    SB.compare_estimators(ours, theirs, X)
    for a, b, (_, _, r) in zip(ours, theirs, problems):
        assert np.array_equal(a.optimizer.gap_hist, b.optimizer.gap_hist)
        assert np.array_equal(a.support_vectors_, b.support_vectors_)
        assert np.array_equal(a.decision_function(X), b.decision_function(X))
        assert a.optimizer.f_x == b.optimizer.f_x and a.optimizer.rho == b.optimizer.rho
        assert np.array_equal(a.optimizer.g_x, b.optimizer.g_x)
    assert conv == conv_theirs
    return ours, theirs


def _same(u, v):
    if isinstance(u, np.ma.MaskedArray) or isinstance(v, np.ma.MaskedArray):
        assert np.array_equal(np.ma.getmaskarray(u), np.ma.getmaskarray(v))
        u, v = np.ma.getdata(u), np.ma.getdata(v)
    if isinstance(u, np.ndarray) and u.dtype.kind == 'f':
        assert u.dtype == v.dtype and np.array_equal(u, v, equal_nan=True)
    else:
        assert len(u) == len(v) and all(a == b for a, b in zip(u, v))


def compare_search(ours, theirs):
    """cv_results_ key for key and value for value (except the *_time keys), the best candidate, the refit"""
    a, b = ours.cv_results_, theirs.cv_results_
    assert list(a) == list(b)
    for key in a:
        if not key.endswith('_time'):
            _same(a[key], b[key])
    for name in ('best_index_', 'best_params_', 'best_score_', 'n_splits_', 'multimetric_'):
        assert hasattr(ours, name) == hasattr(theirs, name)
        if hasattr(ours, name):
            u, v = getattr(ours, name), getattr(theirs, name)
            assert u == v or (u != u and v != v)   # a nan best_score_ when every score is nan
    if hasattr(theirs, 'best_estimator_'):
        SB.compare_estimators([ours.best_estimator_], [theirs.best_estimator_], None)


def sklearn_fits(module):
    """counts the calls of sklearn's _fit_and_score in sklearn.model_selection.<module> (which still runs)"""
    import importlib
    mod = importlib.import_module(f'sklearn.model_selection.{module}')
    return mock.patch.object(mod, '_fit_and_score', wraps=mod._fit_and_score)


def grid_search_both(est, grid, X, y, fit_params=None, shared=True, **kw):
    """this package's GridSearchCV and sklearn's on the same estimator, compared; returns both.  ``shared``: ours
    takes the shared path (else sklearn's own)."""
    from sklearn.model_selection import GridSearchCV as SklearnGrid
    from optiml_b200.model_selection import GridSearchCV
    with warnings.catch_warnings(record=True) as w_ours, sklearn_fits('_search') as fits:
        warnings.simplefilter('always')
        ours = GridSearchCV(est, grid, **kw).fit(X, y, **(fit_params or {}))
    assert (fits.call_count == 0) == shared
    with warnings.catch_warnings(record=True) as w_sk:
        warnings.simplefilter('always')
        theirs = SklearnGrid(est, grid, **kw).fit(X, y, **(fit_params or {}))
    compare_search(ours, theirs)
    conv = [sum(issubclass(x.category, ConvergenceWarning) for x in w) for w in (w_ours, w_sk)]
    assert conv[0] == conv[1]
    return ours, theirs


def cross_validate_both(est, X, y, shared=True, **kw):
    """this package's cross_validate and sklearn's, compared (except the *_time keys); returns ours.  ``shared`` as
    for ``grid_search_both``."""
    from sklearn.model_selection import cross_validate as sklearn_cv
    from optiml_b200.model_selection import cross_validate
    with sklearn_fits('_validation') as fits:
        ours = cross_validate(est, X, y, **kw)
    assert (fits.call_count == 0) == shared
    theirs = sklearn_cv(est, X, y, **kw)
    assert list(ours) == list(theirs)
    for key in ours:
        if key == 'estimator':
            SB.compare_estimators(ours[key], theirs[key], None)
        elif key == 'indices':
            for part in ('train', 'test'):
                assert all(np.array_equal(u, v) for u, v in zip(ours[key][part], theirs[key][part]))
        elif not key.endswith('_time'):
            _same(ours[key], theirs[key])
    return ours


def shared(estimators):
    """the estimators were fitted on shared matrices (not one clone after the other)"""
    return all('batch' in e.fit_times_ for e in estimators)


def check_kkt(est, X, y, rows, tol):
    """the KKT conditions of a fold's SMO solution: the maximal violating pair's gap m - M is below tol, every alpha is
    within its box, and y'alpha = 0 up to rounding"""
    o = est.optimizer
    yv = np.where(y[rows] == est.lb.classes_[1], 1.0, -1.0)
    a, g, C = o.x, o.g_x, est.C
    assert np.all(a >= 0) and np.all(a <= C)
    yg = -yv * g
    up = np.where(yv > 0, a < C, a > 0)
    low = np.where(yv > 0, a > 0, a < C)
    assert yg[up].max() - yg[low].min() < tol
    assert abs(np.dot(yv, a)) <= 1e-9 * max(1.0, np.abs(a).sum())
