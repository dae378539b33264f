"""One-vs-rest / multi-target meta-estimators whose binary problems share one Gram matrix in HBM (SURVEY.md 8f-4).

The reference's multi-class recipe is ``sklearn.multiclass.OneVsRestClassifier(SVC(...))`` (ml/tests/test_svc.py:5,
101-147; ml/svm/_base.py:437-439 tells the user to do so): sklearn clones the estimator once per class and fits the
clones one after the other, so the same n x n Gram matrix is built ``n_classes`` times and every solver streams a
private copy ``Q_c = (y_c y_c') o (K + 1)``.  The classes differ in the label signs only.  The drop-ins below keep
sklearn's contract -- ``estimators_`` holds fitted clones, ``predict`` / ``decision_function`` / ``score`` are
sklearn's own -- but build ``M = K + bias`` ONCE, leave it unsigned, and advance all binary solvers in lockstep with
one streaming pass over M per iteration for up to four problems (``svmb200_pg_run_batch``).  Each clone ends
bit-identical to what ``clone(estimator).fit(X, y_c)`` produces on the same GPU.

``MultiOutputRegressor`` is the same idea for ``SVR``: the targets only change the linear term q.

``optimizer='smo'`` estimators share M too (bias 0, the signs applied on read), but their solvers run side by side on
disjoint ranges of the GPU's SMs (``svmb200_smo_run_batch``) instead of in lockstep: an SMO iteration is bound by
latency, not by bandwidth.  When M would not be resident (``smo.select_row_source`` picks computed rows) the clones are
fitted one after the other, each choosing its own row source.

``fit_shared_gram`` also takes problems on subsets of the rows (the training folds of a grid search,
``optiml_b200/model_selection.py``): SMO then runs each on the matrix of the union of the rows, with the variables
outside its fold held at 0.

Anything the lockstep driver cannot take (a generic callback, ``verbose``, an estimator of another type, fit
parameters, a degenerate class column) goes through sklearn's own ``fit`` -- still on the GPU, one clone after
the other.
"""
import time

import numpy as np
from sklearn import multiclass as _skmc
from sklearn import multioutput as _skmo
from sklearn.base import clone
from sklearn.preprocessing import LabelBinarizer

from .svm._base import SVC, SVR
from .svm.smo import SMO
from .svm.kernels import _dense_f64
from ..opti.batch import minimize_batch

__all__ = ['OneVsRestClassifier', 'MultiOutputRegressor', 'fit_shared_gram']


def fit_shared_gram(estimator, X, problems):
    """Fit one clone of ``estimator`` (an ``SVC`` or ``SVR`` of this package on the dual path) per problem on resident
    Gram matrices shared between problems.  A problem is ``(params, target, rows)``: the clone is
    ``clone(estimator).set_params(**params)``, fitted on ``X[rows]`` and ``target`` (the labels / targets of those rows;
    ``rows=None``: every row of X).  One-vs-rest and multi-target fits are the case "every row, no params".

    Problems whose clones resolve the same kernel spec share ONE matrix, built on the union of their rows (kept in index
    order, so that a problem's part of it is bit for bit the matrix of its own rows: K1 computes every element from its
    two samples alone).  ``gamma='scale'`` depends on the rows, so such problems share only with problems on the same
    rows.  A problem on a proper subset of the union runs on its variables only (``SMO`` with ``active``).

    Returns the fitted clones in the order of ``problems``; each reports in ``fit_times_`` the number of problems that
    shared its matrix (``batch``) and its share of the wall clock of its group (``share_s``: the group's wall clock
    divided by its problems)."""
    if not isinstance(estimator, (SVC, SVR)):
        raise TypeError(f'{estimator} is not an SVC / SVR of optiml_b200')
    problems = [(params or {}, np.asarray(t), None if r is None else np.asarray(r, dtype=np.int64))
                for params, t, r in problems]
    if not problems:
        return []
    clones = [clone(estimator).set_params(**clone(params, safe=False)) for params, _, _ in problems]
    X, _ = _dense_f64(X, None, finite=False)  # the all-finite test runs on the device copy (_build_hessian)
    groups = {}
    for k, (est, (_, _, rows)) in enumerate(zip(clones, problems)):
        # rows out of ascending order: the clone's matrix is not a part of one in index order, so it is fitted alone
        own = rows is not None and np.any(np.diff(rows) <= 0)
        groups.setdefault(('own', k) if own else _gram_key(est, X.shape[1], rows), []).append(k)
    for members in groups.values():
        _fit_group([clones[k] for k in members], [problems[k][1:] for k in members], X)
    return clones


def _gram_key(est, d, rows):
    """What a clone's Gram matrix depends on besides the rows: the kernel spec as the clone resolves it (gamma='scale'
    from the variance of its own rows: no sharing across row sets), and the layout"""
    kernel, layout = est.kernel, 'svr' if isinstance(est, SVR) else 'plain'
    if getattr(kernel, 'gamma', None) == 'scale':
        gamma = ('scale', None if rows is None else rows.tobytes())
    else:
        gamma = float(kernel.resolve_gamma(np.empty((0, d))))
    return (layout, kernel.kernel_id, gamma, float(getattr(kernel, 'coef0', 0.)), float(getattr(kernel, 'degree', 1)),
            est._bias())


def _fit_group(clones, problems, X):
    """``fit_shared_gram`` for problems with one kernel spec: on one matrix when ``_fit_on_one_gram`` can, else one
    clone after the other"""
    t0 = time.perf_counter()
    if not _fit_on_one_gram(clones, problems, X):
        for est, (t, rows) in zip(clones, problems):
            est.fit(X if rows is None else X[rows], t)
    share_s = (time.perf_counter() - t0) / len(clones)
    for est in clones:
        est.fit_times_['share_s'] = share_s


def _fit_on_one_gram(clones, problems, X):
    """K1 once on the union of the problems' rows, every solver in one batch, every clone finished.  False, before any
    device work, when a clone fits alone (rows in an order of their own) or SMO would not keep M resident."""
    head = clones[0]
    layout = 'svr' if isinstance(head, SVR) else 'plain'
    union, Xu = None, X
    if any(rows is not None for _, rows in problems):
        problems = [(t, np.arange(len(X)) if rows is None else rows) for t, rows in problems]
        union = np.unique(np.concatenate([rows for _, rows in problems]))
        Xu = X if len(union) == len(X) else X[union]
    if union is not None and len(problems) == 1 and np.any(np.diff(problems[0][1]) <= 0):
        return False
    if head._bcqp_solver_class() is SMO:  # (raises for the branches outside the dual path before any device work)
        n, d = Xu.shape
        head._check_solver_scope(SMO, n)
        if head._smo_row_source(n, d, layout)[0] != 'resident':
            return False
    # K1 once: M = K + bias without label signs (SVC: the solvers apply them; SVR: the block signs are implicit)
    shared = head._build_hessian(Xu, None, layout, None, head._bias())
    gram_s = head.fit_times_['gram_s']
    dX, owned = head._train_X_device   # every clone gathers its support vectors from this one copy of X in HBM
    try:
        plans = []
        for est, (t, rows) in zip(clones, problems):
            if union is None:
                plans.append(est._plan_fit(X, t, shared=shared))
            else:   # the problem's rows are these rows of M (whose rows are the union, ascending)
                plans.append(est._plan_fit(X[rows], t, shared=shared, rows=np.searchsorted(union, rows)))
        t0 = time.perf_counter()
        minimize_batch([p['solver'] for p in plans])
        solve_s = time.perf_counter() - t0
        for est, plan in zip(clones, plans):
            # wall-clock of the shared steps: every clone reports the whole batch
            est.fit_times_ = {'gram_s': gram_s, 'solve_s': solve_s, 'batch': len(clones)}
            est._train_X_device = (dX, False)
            est._finish_fit(plan)
    finally:
        for est in clones:
            est._train_X_device = None
        if owned:
            dX.release()
    return True


def _smo_batch_capable(estimator):
    """An ``optimizer='smo'`` estimator whose clones ``fit_shared_gram`` can run as one SMO batch: nothing on the host
    watches the solve.  (Sharded fits raise in ``fit_shared_gram``, as they do in a single fit.)"""
    if not isinstance(estimator, (SVC, SVR)) or estimator.verbose:
        return False
    try:
        return estimator._bcqp_solver_class() is SMO
    except (NotImplementedError, TypeError, ValueError):   # (ValueError: shrinking without SMO, refused at fit)
        return False


def _lockstep_capable(estimator, n_samples=None):
    """The estimator runs a device-resident solver that nothing on the host has to watch (and the problem is not one a
    single-process device group shards over its GPUs: there the clones are fitted one after the other, each on all GPUs)."""
    if not isinstance(estimator, (SVC, SVR)) or estimator.verbose:
        return False
    if n_samples is not None:
        from ..runtime import default_context
        group = default_context().group
        if group is not None and group.wants(int(n_samples)):
            return False
    try:
        solver_cls = estimator._bcqp_solver_class()
    except (NotImplementedError, TypeError, ValueError):   # (ValueError: shrinking without SMO, refused at fit)
        return False
    return solver_cls is not SMO   # SMO batches are not lockstep ones: _smo_batch_capable


class OneVsRestClassifier(_skmc.OneVsRestClassifier):
    """``sklearn.multiclass.OneVsRestClassifier`` whose binary ``SVC`` problems share one Gram matrix."""

    def fit(self, X, y, **fit_params):
        if fit_params or not isinstance(self.estimator, SVC) or \
                not (_lockstep_capable(self.estimator, np.shape(X)[0]) or _smo_batch_capable(self.estimator)):
            return super().fit(X, y, **fit_params)
        self._validate_params()
        # label handling of sklearn/multiclass.py OneVsRestClassifier.fit
        label_binarizer = LabelBinarizer(sparse_output=True)
        Y = label_binarizer.fit_transform(y).tocsc()
        columns = [col.toarray().ravel() for col in Y.T]
        if len(columns) < 2 or any(len(np.unique(c)) == 1 for c in columns):
            return super().fit(X, y)  # a single problem, or a constant column (sklearn's _ConstantPredictor)
        self.label_binarizer_ = label_binarizer
        self.classes_ = label_binarizer.classes_
        self.estimators_ = fit_shared_gram(self.estimator, X, [({}, c, None) for c in columns])
        if hasattr(self.estimators_[0], 'n_features_in_'):
            self.n_features_in_ = self.estimators_[0].n_features_in_
        if hasattr(self.estimators_[0], 'feature_names_in_'):
            self.feature_names_in_ = self.estimators_[0].feature_names_in_
        return self


class MultiOutputRegressor(_skmo.MultiOutputRegressor):
    """``sklearn.multioutput.MultiOutputRegressor`` whose per-target ``SVR`` problems share one Gram matrix."""

    def fit(self, X, y, sample_weight=None, **fit_params):
        y_arr = np.asarray(y)
        if sample_weight is not None or fit_params or not isinstance(self.estimator, SVR) or \
                not (_lockstep_capable(self.estimator, np.shape(X)[0]) or _smo_batch_capable(self.estimator)) or \
                y_arr.ndim != 2 or y_arr.shape[1] < 2:
            return super().fit(X, y, sample_weight=sample_weight, **fit_params)
        self._validate_params()
        self.estimators_ = fit_shared_gram(self.estimator, X, [({}, y_arr[:, i], None) for i in range(y_arr.shape[1])])
        if hasattr(self.estimators_[0], 'n_features_in_'):
            self.n_features_in_ = self.estimators_[0].n_features_in_
        if hasattr(self.estimators_[0], 'feature_names_in_'):
            self.feature_names_in_ = self.estimators_[0].feature_names_in_
        return self
