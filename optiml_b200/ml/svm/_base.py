"""sklearn-compatible SVM estimators for the dual, box-constrained formulation, trained on the GPU.

Host mirror of optiml/ml/svm/_base.py restricted to the branch
``dual=True, reg_intercept=True, loss in {hinge, epsilon_insensitive}, optimizer=<BCQP solver>``,
its augmented-Lagrangian relaxation (``optimizer=<StochasticOptimizer>``) and SMO for the dual with
its equality constraint (``optimizer='smo', reg_intercept=False``, ml/svm/smo.py):
same constructor keywords (sklearn ``clone``/``get_params`` work), same validation errors, same
fitted attributes.  Every other branch of the reference (primal losses, other string QP solvers,
plain Lagrangian duals) raises ``NotImplementedError`` -- they are different algorithms and out of scope.

Where the reference builds K, Q = K o yy' + yy' and three more n x n temporaries on the host
(ml/svm/_base.py:552-554, 628; opti/_base.py:243), here the Hessian is produced directly in HBM by
the fused Gram kernel, row-sharded over the GPUs of the job, and never visits the host.
"""
import ctypes as C
import warnings

import numpy as np
from sklearn.base import BaseEstimator, ClassifierMixin, RegressorMixin
from sklearn.exceptions import ConvergenceWarning
from sklearn.preprocessing import LabelBinarizer

from .kernels import gaussian, Kernel, LinearKernel, _dense_f64, gather_rows
from .smo import SMO, select_row_source
from .losses import (squared_hinge, squared_epsilon_insensitive, Hinge, SquaredHinge, EpsilonInsensitive,
                     SquaredEpsilonInsensitive)
from ... import _native as N
from ...opti import Optimizer, Quadratic
from ...opti.constrained import AugmentedLagrangianQuadratic, BoxConstrainedQuadraticOptimizer, ProjectedGradient
from ...opti.unconstrained.stochastic import StochasticOptimizer, StochasticMomentumOptimizer
from ...runtime import (DeviceHessian, DeviceMatrix, GroupHessian, KernelRowsHessian, default_context, make_hessian,
                       would_shard)

_SCOPE = ('optiml_b200 implements the dual formulation solved by a BoxConstrainedQuadraticOptimizer '
          '(ProjectedGradient, FrankWolfe; reg_intercept=True) or, as its augmented-Lagrangian relaxation, by a '
          'StochasticOptimizer (AdaGrad, ...); {} is outside that path')


def _embed(nvars, cols, *vectors):
    """A problem on the variables ``cols`` of a shared matrix with ``nvars`` variables: each vector spread to its
    columns (1 elsewhere: a valid sign, never read as a bound or a linear term), and the mask of the active variables"""
    out = []
    for v in vectors:
        full = np.ones(nvars)
        full[cols] = v
        out.append(full)
    active = np.zeros(nvars, dtype=bool)
    active[cols] = True
    return out, active


def _binarize(lb, y):
    """``lb.transform(y).ravel()`` for the labels ``lb`` was just fitted on (ml/svm/_base.py:440).  For a plain
    two-class 1-D target LabelBinarizer's answer is written down directly (int64, classes_[1] -> +1, classes_[0] -> -1):
    its sparse-matrix detour costs 7 ms at n = 50 000 on every rank of a sharded fit."""
    ya = np.asarray(y)
    if ya.ndim == 1 and len(lb.classes_) == 2 and lb.y_type_ == 'binary':
        # label_binarize keeps a signed-integer label dtype and uses the index dtype otherwise
        dt = ya.dtype if np.issubdtype(ya.dtype, np.signedinteger) else np.intp
        return np.where(ya == lb.classes_[1], 1, -1).astype(dt, copy=False)
    return lb.transform(y).ravel()


class SVM(BaseEstimator):
    """Common constructor / decision function (optiml/ml/svm/_base.py:26-293)."""

    def __init__(self, loss=None, kernel=gaussian, C=1, rho=1, mu=1, fit_intercept=True, intercept_scaling=1,
                 reg_intercept=False, dual=False, optimizer=None, master_solver='clarabel', learning_rate='auto',
                 momentum_type='none', momentum=0.9, max_iter=1000, max_f_eval=15000, tol=1e-4, batch_size=None,
                 shuffle=True, random_state=None, early_stopping=False, validation_split=0., patience=5,
                 verbose=False, master_verbose=False, shrinking=False):
        self.loss = loss
        if not isinstance(kernel, Kernel):
            raise TypeError(f'{kernel} is not an allowed kernel function')
        self.kernel = kernel
        if not C > 0:
            raise ValueError('C must be > 0')
        self.C = C
        if not rho > 0:
            raise ValueError('rho must be > 0')
        self.rho = rho
        if not mu > 0:
            raise ValueError('mu must be > 0')
        self.mu = mu
        if not isinstance(fit_intercept, bool):
            raise ValueError('fit_intercept mu be a boolean value')
        self.fit_intercept = fit_intercept
        self.intercept_scaling = intercept_scaling
        if not isinstance(reg_intercept, bool):
            raise ValueError('reg_intercept mu be a boolean value')
        self.reg_intercept = reg_intercept
        if not isinstance(dual, bool):
            raise ValueError('dual must be a boolean value')
        self.dual = dual
        if not self.dual and not (isinstance(optimizer, type) and issubclass(optimizer, Optimizer)) \
                and optimizer is not None:
            raise TypeError(f'{optimizer} is not an allowed optimization method')
        self.optimizer = optimizer
        self.master_solver = master_solver
        self.learning_rate = learning_rate
        self.max_iter = max_iter
        self.max_f_eval = max_f_eval
        self.momentum_type = momentum_type
        self.momentum = momentum
        if not tol > 0:
            raise ValueError('tol must be > 0')
        self.tol = tol
        self.batch_size = batch_size
        self.shuffle = shuffle
        self.random_state = random_state
        self.early_stopping = early_stopping
        self.validation_split = validation_split
        self.patience = patience
        self.verbose = verbose
        self.master_verbose = master_verbose
        self.shrinking = shrinking   # libsvm's shrinking heuristic (optimizer='smo' only; checked at fit)
        if not self.dual or isinstance(self.kernel, LinearKernel):
            self.coef_ = np.zeros(0)
        self.intercept_ = 0.
        self.support_ = np.zeros(0)
        self._sv_device = None
        self.support_vectors_ = np.zeros(0)
        if self.dual:
            self.alphas_ = np.zeros(0)
            self.dual_coef_ = np.zeros(0)
        if not isinstance(optimizer, str):
            self.train_loss_history = []

    # ------------------------------------------------------------------ shared pieces of fit
    def _bcqp_solver_class(self):
        solver_cls = self._bcqp_solver_class_of_optimizer()
        if getattr(self, 'shrinking', False) and solver_cls is not SMO:
            raise ValueError("shrinking=True is libsvm's heuristic for the SMO solver: it needs optimizer='smo'")
        return solver_cls

    def _bcqp_solver_class_of_optimizer(self):
        """The solver class to instantiate; mirrors the dispatch of ml/svm/_base.py:559-725.  A
        ``StochasticOptimizer`` subclass selects the augmented-Lagrangian relaxation (:638-723), ``'smo'`` the SMO
        solver of the problem with its equality constraint (ml/svm/smo.py)."""
        opt = self.optimizer
        if isinstance(opt, (BoxConstrainedQuadraticOptimizer, StochasticOptimizer)):
            opt = type(opt)  # refit of an estimator whose ``optimizer`` was replaced by the fitted instance
        if isinstance(opt, SMO):
            opt = 'smo'
        if not self.dual:
            raise NotImplementedError(_SCOPE.format('dual=False (primal formulation)'))
        if isinstance(opt, str) and opt == 'smo':
            if self.reg_intercept:
                raise NotImplementedError("optimizer='smo' solves the dual with the equality constraint of an "
                                          "unregularised intercept (reg_intercept=False); with reg_intercept=True there "
                                          "is no such constraint: use ProjectedGradient or FrankWolfe")
            return SMO
        if isinstance(opt, str) or opt is None:
            raise NotImplementedError(_SCOPE.format(f'optimizer={opt!r}'))
        if isinstance(opt, type) and issubclass(opt, StochasticOptimizer):
            return opt
        if not (isinstance(opt, type) and issubclass(opt, BoxConstrainedQuadraticOptimizer)):
            raise NotImplementedError(_SCOPE.format(f'optimizer={opt}'))
        if not self.reg_intercept:
            # ml/svm/_base.py:621-624, 1171-1174: no BCQP solver handles the equality constraint
            raise NotImplementedError
        return opt

    def _make_solver(self, solver_cls, hessian, q, ub, eq_row, active=None):
        """The selected solver, ready to run, on  min x'Qx/2 + q'x : 0 <= x <= ub (, eq_row'x = 0 when the intercept
        is not regularised); sets ``self.obj`` like ml/svm/_base.py:628-725.  ``active``: SMO on these variables only
        (``_embed``)."""
        if solver_cls is SMO:
            # no callback: for a string optimizer there is no train_loss_history (SVM.__init__); the histories stay
            # on the solver
            self.obj = Quadratic(hessian, q)
            return SMO(quad=self.obj, y=eq_row, C=ub, tol=self.tol, max_iter=self.max_iter, verbose=self.verbose,
                       active=active, shrinking=bool(getattr(self, 'shrinking', False)))
        if active is not None:
            raise ValueError("a problem on a subset of a shared matrix's rows needs optimizer='smo'")
        if issubclass(solver_cls, BoxConstrainedQuadraticOptimizer):
            self.obj = Quadratic(hessian, q)
            solver = solver_cls(quad=self.obj, ub=ub, tol=self.tol, max_iter=self.max_iter,
                                callback=self._store_train_info, verbose=self.verbose)
            solver.profile = bool(getattr(self, 'profile_matvec', False))  # CUDA events around every K2 launch
            return solver
        # augmented-Lagrangian relaxation of the box (and of the equality), ml/svm/_base.py:638-655, 1188-1205
        lb = np.zeros_like(ub)
        if self.reg_intercept:
            self.obj = AugmentedLagrangianQuadratic(primal=Quadratic(hessian, q), lb=lb, ub=ub, rho=self.rho)
        else:
            self.obj = AugmentedLagrangianQuadratic(primal=Quadratic(hessian, q), A=eq_row, b=np.zeros(1), lb=lb,
                                                    ub=ub, rho=self.rho)
        kwargs = dict(f=self.obj, tol=self.tol, step_size=self.learning_rate, epochs=self.max_iter,
                      random_state=self.random_state, callback=self._store_train_info, verbose=self.verbose)
        if issubclass(solver_cls, StochasticMomentumOptimizer):
            kwargs.update(momentum_type=self.momentum_type, momentum=self.momentum)
        solver = solver_cls(**kwargs)
        solver.profile = bool(getattr(self, 'profile_matvec', False))
        return solver

    def _after_solver(self, solver):
        if isinstance(solver, (StochasticOptimizer, SMO)) and solver.status == 'stopped':  # ml/svm/_base.py:715-717
            warnings.warn('max_iter reached but the optimization has not converged yet', ConvergenceWarning)

    @staticmethod
    def _check_solver_scope(solver_cls, n):
        """SMO holds the whole Hessian on one GPU: refuse, before any device work, a fit whose matrix would be sharded."""
        if solver_cls is SMO and would_shard(n):
            raise NotImplementedError("optimizer='smo' runs on one GPU: this fit would shard its Hessian over several "
                                      "(torchrun world > 1, or a device group)")

    def _bias(self):
        """The Hessian carries the rank-one term yy' (SVC) / ee' (SVR) only when the intercept is regularised
        (ml/svm/_base.py:628, 652 vs 644; 1178, 1202 vs 1194)."""
        return 1.0 if self.reg_intercept else 0.0

    def _build_hessian(self, X, signs, layout, X_device=None, bias=1.0):
        """K1: Gram matrix + bias (+ label signs) straight into this rank's row shard in HBM.
        ``X_device`` (a DeviceMatrix already holding X) skips the host->device copy of X."""
        import time
        ctx = default_context()
        n, d = X.shape
        t0 = time.perf_counter()
        dX = X_device if X_device is not None else ctx.upload_matrix(X)
        # gamma='scale' needs X.var(), the input validation an all-finite test: both from the copy in HBM, one pass
        kid, gamma, coef0, degree = self.kernel.gram_spec(X, device=dX)
        H = make_hessian(ctx, n, layout)
        if isinstance(H, GroupHessian):
            # one process, N GPUs: X is replicated over NVLink, every rank builds its row shard, all at once
            copies = ctx.group.replicate(dX)
            sign_copies = [c.upload_vector(signs) if signs is not None else None for c in ctx.group.ctxs]
            for part, dXr, dSr in zip(H.parts, copies, sign_copies):
                sp = C.c_void_p(dSr.dptr) if dSr is not None else None
                N.call('svmb200_gram', part.ctx.handle, C.c_void_p(dXr.dptr), n, dXr.ld, C.c_void_p(dXr.dptr), n, dXr.ld, d, 1,
                       kid, gamma, coef0, degree, sp, sp, float(bias), part.row0, part.nrows, C.c_void_p(part.matrix.dptr),
                       part.ld)
                part.matrix.self_gram = True
            ctx.group.sync()
            for m in copies + [v for v in sign_copies if v is not None]:
                m.release()
        else:
            dS = ctx.upload_vector(signs) if signs is not None else None
            sp = C.c_void_p(dS.dptr) if dS is not None else None
            N.call('svmb200_gram', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, C.c_void_p(dX.dptr), n, dX.ld, d, 1, kid,
                   gamma, coef0, degree, sp, sp, float(bias), H.row0, H.nrows, C.c_void_p(H.matrix.dptr), H.ld)
            H.matrix.self_gram = True
            ctx.sync()
            if dS is not None:
                dS.release()
        # X stays in HBM until the support vectors have been gathered from it (_set_support_vectors)
        self._train_X_device = (dX, X_device is None)
        self.fit_times_ = {'gram_s': time.perf_counter() - t0}  # gamma + upload + Gram kernel (wall clock)
        return H

    @staticmethod
    def _smo_row_source(n, d, layout):
        """``smo.select_row_source`` for an SMO fit of n samples with d features started now."""
        ctx = default_context()
        info = ctx.info()
        info['free_bytes'] += ctx.pooled_bytes()   # parked buffers are given back when an allocation needs them
        return select_row_source(n, 2 * n if layout == 'svr' else n, N.padded_ld(n), d, info)

    def _smo_hessian(self, X, signs, layout, X_device=None):
        """SMO's Hessian: resident (K1, as for the other solvers) when it fits in the free device memory, else computed
        rows (K12: no matrix, rows from X on the device, with a row cache) -- chosen by smo.select_row_source before
        any device work."""
        import time
        ctx = default_context()
        n, d = X.shape
        source, cache_bytes = self._smo_row_source(n, d, layout)
        if source == 'resident':
            return self._build_hessian(X, signs, layout, X_device, 0.0)
        ctx.trim()   # the row cache is allocated by the solver, outside the pool
        t0 = time.perf_counter()
        dX = X_device if X_device is not None else ctx.upload_matrix(X)
        spec = self.kernel.gram_spec(X, device=dX)
        if X_device is not None:   # the Hessian owns its reference to X: a private copy of the caller's matrix
            own = DeviceMatrix(ctx, dX.rows, dX.cols, dX.ld)
            N.call('svmb200_d2d', ctx.handle, C.c_void_p(own.dptr), C.c_void_p(dX.dptr), dX.nbytes)
            dX = own
        H = KernelRowsHessian(ctx, dX, X, spec, layout, signs, cache_bytes)
        # the support vectors are gathered from the Hessian's X, which it frees on release (_set_support_vectors)
        self._train_X_device = (dX, False)
        self.fit_times_ = {'gram_s': time.perf_counter() - t0}  # gamma + upload (no Gram matrix is built)
        return H

    # ------------------------------------------------------------------ support vectors: device-resident, host copy on demand
    @property
    def support_vectors_(self):
        """``X[support_]`` (ml/svm/_base.py:869, 1425).  After a kernelised fit the rows are gathered in HBM, where
        ``decision_function`` needs them, from the copy of X the fit uploaded -- a snapshot of the training data at fit
        time, like the reference's; the host array is materialised on first access (50 MB at n = 50 000, d = 128: the
        copy into fresh host memory alone was 8 ms of every fit on every rank)."""
        if self._sv_host is None and self._sv_device is not None:
            self._sv_host = self._sv_device.to_host()
        return self._sv_host

    @support_vectors_.setter
    def support_vectors_(self, value):
        self._sv_host, self._sv_device = value, None

    def _set_support_vectors(self, X, rows=None):
        """``rows``: the rows of the device copy of X that X's rows are (a fold's training rows in a shared matrix)"""
        dX, owned = getattr(self, '_train_X_device', None) or (None, False)
        self._train_X_device = None
        if dX is not None and dX.dptr and not isinstance(self.kernel, LinearKernel) and len(self.support_):
            ctx = dX.ctx
            idx = np.ascontiguousarray(self.support_ if rows is None else rows[self.support_], dtype=np.int64)
            sv = DeviceMatrix(ctx, len(idx), dX.cols, dX.ld)
            N.call('svmb200_gather_rows', ctx.handle, C.c_void_p(dX.dptr), dX.rows, dX.ld, dX.cols,
                   idx.ctypes.data_as(C.c_void_p), len(idx), C.c_void_p(sv.dptr), sv.ld)
            self._sv_host, self._sv_device = None, sv
        else:
            self.support_vectors_ = gather_rows(X, self.support_)
        if dX is not None and owned:
            dX.release()

    def __getstate__(self):
        """Fitted estimators pickle / deep-copy without device handles: the support vectors travel as the host array."""
        state = super().__getstate__()
        if state.get('_sv_device') is not None:
            state['_sv_host'] = self.support_vectors_
        state['_sv_device'] = None
        state['_train_X_device'] = None
        return state

    def decision_function(self, X):
        """ml/svm/_base.py:284-287.  ``gamma='scale'`` is resolved from ``support_vectors_`` (the first
        argument of the reference's kernel call), not from the training matrix."""
        if self.dual and not isinstance(self.kernel, LinearKernel) and self._sv_device is not None and self._sv_device.dptr:
            # support vectors already in HBM (left there by fit): no upload, gamma='scale' from the device copy
            X, _ = _dense_f64(X, None)
            dsv = self._sv_device
            coef = np.ascontiguousarray(self.dual_coef_, dtype=np.float64)
            kid, gamma, coef0, degree = self.kernel.gram_spec(None, device=dsv)
            out = np.empty(X.shape[0])
            N.call('svmb200_decision_device', dsv.ctx.handle, C.c_void_p(dsv.dptr), dsv.rows, dsv.ld, N.ptr(coef), N.ptr(X),
                   X.shape[0], X.shape[1], kid, gamma, coef0, degree, float(self.intercept_), N.ptr(out))
            return out
        if self.dual and not isinstance(self.kernel, LinearKernel):
            X, _ = _dense_f64(X, None)
            sv = np.ascontiguousarray(self.support_vectors_, dtype=np.float64)
            coef = np.ascontiguousarray(self.dual_coef_, dtype=np.float64)
            kid, gamma, coef0, degree = self.kernel.gram_spec(sv)
            out = np.empty(X.shape[0])
            N.call('svmb200_decision', default_context().handle, N.ptr(sv), sv.shape[0], N.ptr(coef), N.ptr(X),
                   X.shape[0], X.shape[1], kid, gamma, coef0, degree, float(self.intercept_), N.ptr(out))
            return out
        # linear dual / primal form X @ coef_ + b (ml/svm/_base.py:287): streaming matvec over the rows of X
        X, _ = _dense_f64(X, None)
        ctx = default_context()
        dX = ctx.upload_matrix(X)
        dcoef = ctx.upload_vector(self.coef_, length=dX.ld)
        dout = ctx.malloc(8 * X.shape[0])
        out = np.empty(X.shape[0])
        try:
            N.call('svmb200_matvec', ctx.handle, C.c_void_p(dX.dptr), X.shape[0], dX.ld, C.c_void_p(dcoef.dptr),
                   C.c_void_p(dout))
            ctx.d2h(out, dout)
        finally:
            ctx.free(dout)
            dX.release()
            dcoef.release()
        return out + self.intercept_

    def _store_train_info(self, opt):
        # ml/svm/_base.py:289-293
        self.train_loss_history.append(opt.primal_f_x if opt.is_lagrangian_dual() else opt.f_x)

    _store_train_info._svmb200_history_only = True


class SVC(ClassifierMixin, SVM):
    """C-Support Vector Classification, dual hinge-loss problem (optiml/ml/svm/_base.py:354-885)."""

    def __init__(self, loss=squared_hinge, kernel=gaussian, C=1, rho=1, mu=1, fit_intercept=True,
                 intercept_scaling=1, reg_intercept=False, dual=False, optimizer=None, master_solver='clarabel',
                 learning_rate='auto', momentum_type='none', momentum=0.9, max_iter=1000, max_f_eval=15000, tol=1e-4,
                 batch_size=None, shuffle=True, random_state=None, early_stopping=False, validation_split=0.,
                 patience=5, verbose=False, master_verbose=False, shrinking=False):
        super(SVC, self).__init__(loss=loss, kernel=kernel, C=C, rho=rho, mu=mu, fit_intercept=fit_intercept,
                                  intercept_scaling=intercept_scaling, reg_intercept=reg_intercept, dual=dual,
                                  optimizer=optimizer, master_solver=master_solver, learning_rate=learning_rate,
                                  momentum_type=momentum_type, momentum=momentum, max_iter=max_iter,
                                  max_f_eval=max_f_eval, tol=tol, batch_size=batch_size, shuffle=shuffle,
                                  random_state=random_state, early_stopping=early_stopping,
                                  validation_split=validation_split, patience=patience, verbose=verbose,
                                  master_verbose=master_verbose, shrinking=shrinking)
        if not getattr(loss, '_loss_type', None) == 'classifier':
            raise TypeError(f'{loss} is not an allowed SVC loss function')
        self.lb = LabelBinarizer(neg_label=-1)

    def fit(self, X, y, X_device=None):
        import time
        plan = self._plan_fit(X, y, X_device)
        t0 = time.perf_counter()
        plan['solver'].minimize()
        self.fit_times_['solve_s'] = time.perf_counter() - t0
        return self._finish_fit(plan)

    def _plan_fit(self, X, y, X_device=None, shared=None, rows=None):
        """Everything ``fit`` does before the solver runs.  ``shared``: an unsigned resident ``M = K + bias`` that other
        binary problems on the same X use too (one-vs-rest, ml/multiclass.py); the label signs are then applied by
        the solver instead of being baked into a private copy of Q.  ``rows``: X and y are the rows ``rows`` (ascending)
        of the set M was built on -- a cross-validation fold; the solver runs on those variables only (``_embed``)."""
        self.lb.fit(y)
        if len(self.lb.classes_) > 2:
            raise ValueError('use OneVsOneClassifier or OneVsRestClassifier from sklearn.multiclass '
                             'to train a model over more than two labels')
        y = _binarize(self.lb, y)
        solver_cls = self._bcqp_solver_class()
        self._check_solver_scope(solver_cls, len(y))
        if self.loss == SquaredHinge:
            raise NotImplementedError  # ml/svm/_base.py:771-774
        if self.loss != Hinge:
            raise TypeError(f'{self.loss} is not an allowed loss')
        X, _ = _dense_f64(X, None, finite=False)  # the all-finite test runs on the device copy (_build_hessian)
        n = len(y)
        ys = y.astype(np.float64)

        # Q = K o yy' (+ yy' when the intercept is regularised)  (ml/svm/_base.py:552-554, 628), q = -1, 0 <= alpha <= C
        bias = self._bias()
        ub, q, eq, active = np.ones(n) * self.C, -np.ones(n), y, None
        if shared is not None:
            signs = ys
            if rows is not None:
                (signs, q, ub), active = _embed(shared.n, rows, ys, q, ub)
                eq = signs
            hessian = shared.with_signs(signs)
            self.fit_times_ = {}
        elif solver_cls is SMO:
            hessian = self._smo_hessian(X, ys, 'plain', X_device)
        else:
            hessian = self._build_hessian(X, ys, 'plain', X_device, bias)
        solver = self._make_solver(solver_cls, hessian, q, ub, eq, active)
        return dict(X=X, y=y, ys=ys, n=n, bias=bias, solver=solver, rows=rows)

    def _finish_fit(self, plan):
        """Everything ``fit`` does after the solver has run (ml/svm/_base.py:725, 867-880)."""
        X, y, ys, n, bias = plan['X'], plan['y'], plan['ys'], plan['n'], plan['bias']
        self.optimizer = plan['solver']
        self._after_solver(self.optimizer)
        self.alphas_ = self.optimizer.x

        # support set, dual coefficients, intercept (ml/svm/_base.py:867-880)
        sv = self.alphas_ > 1e-6
        self.support_ = np.arange(n)[sv]
        self._set_support_vectors(X, plan['rows'])
        sv_y, alphas = y[sv], self.alphas_[sv]
        self.dual_coef_ = alphas * sv_y
        if isinstance(self.kernel, LinearKernel):
            self.coef_ = np.dot(self.dual_coef_, self.support_vectors_)
        if isinstance(self.optimizer, SMO):
            self.intercept_ = -self.optimizer.rho   # libsvm's intercept from the final alpha and G
            return self
        # K5: sum_m dual_coef_m K[n, m] for every n from ONE masked pass over the resident
        # Q = s_n s_m (K + bias):  s_n (Q beta)_n = sum_m dual_coef_m K[n, m] + bias sum_m dual_coef_m
        v = self.obj.device_hessian().product(np.where(sv, self.alphas_, 0.))
        k_dot = ys[sv] * v[sv] - bias * np.sum(self.dual_coef_)
        self.intercept_ = float(np.sum(sv_y - k_dot)) / len(alphas)
        return self

    def predict(self, X):
        return self.lb.inverse_transform(self.decision_function(X))


class SVR(RegressorMixin, SVM):
    """Epsilon-Support Vector Regression, dual eps-insensitive problem (ml/svm/_base.py:888-1442)."""

    def __init__(self, loss=squared_epsilon_insensitive, epsilon=0.1, kernel=gaussian, C=1, rho=1, mu=1,
                 fit_intercept=True, intercept_scaling=1, reg_intercept=False, dual=False, optimizer=None,
                 master_solver='clarabel', learning_rate='auto', momentum_type='none', momentum=0.9, max_iter=1000,
                 max_f_eval=15000, tol=1e-4, batch_size=None, shuffle=True, random_state=None, early_stopping=False,
                 validation_split=0., patience=5, verbose=False, master_verbose=False, shrinking=False):
        super(SVR, self).__init__(loss=loss, kernel=kernel, C=C, rho=rho, mu=mu, fit_intercept=fit_intercept,
                                  intercept_scaling=intercept_scaling, reg_intercept=reg_intercept, dual=dual,
                                  optimizer=optimizer, master_solver=master_solver, learning_rate=learning_rate,
                                  momentum_type=momentum_type, momentum=momentum, max_iter=max_iter,
                                  max_f_eval=max_f_eval, tol=tol, batch_size=batch_size, shuffle=shuffle,
                                  random_state=random_state, early_stopping=early_stopping,
                                  validation_split=validation_split, patience=patience, verbose=verbose,
                                  master_verbose=master_verbose, shrinking=shrinking)
        if not getattr(loss, '_loss_type', None) == 'regressor':
            raise TypeError(f'{loss} is not an allowed SVR loss function')
        if not epsilon >= 0:
            raise ValueError('epsilon must be >= 0')
        self.epsilon = epsilon

    def fit(self, X, y, X_device=None):
        import time
        plan = self._plan_fit(X, y, X_device)
        t0 = time.perf_counter()
        plan['solver'].minimize()
        self.fit_times_['solve_s'] = time.perf_counter() - t0
        return self._finish_fit(plan)

    def _plan_fit(self, X, y, X_device=None, shared=None, rows=None):
        """Everything ``fit`` does before the solver runs.  ``shared``: the resident ``M = K + bias`` of another
        regression on the same X (multi-target fits, ml/multiclass.py) -- targets only change q.  ``rows``: as for
        ``SVC._plan_fit``."""
        y = np.asarray(y)
        targets = y.shape[1] if y.ndim > 1 else 1
        if targets > 1:
            raise ValueError('use sklearn.multioutput.MultiOutputRegressor '
                             'to train a model over more than one target')
        solver_cls = self._bcqp_solver_class()
        self._check_solver_scope(solver_cls, len(y))
        if self.loss == SquaredEpsilonInsensitive:
            raise NotImplementedError  # ml/svm/_base.py:1325-1328
        if self.loss != EpsilonInsensitive:
            raise TypeError(f'{self.loss} is not an allowed loss')
        X, _ = _dense_f64(X, None, finite=False)  # the all-finite test runs on the device copy (_build_hessian)
        y = y.astype(np.float64).ravel()
        n = len(y)

        # Q = [[K, -K], [-K, K]] (+ ee', e = [1, -1], when the intercept is regularised)  (ml/svm/_base.py:1098-1100,
        # 1126, 1178): only M = K + bias (n x n) is resident, the solver applies the block signs
        bias = self._bias()
        ub, q, e, active = np.ones(2 * n) * self.C, np.hstack((-y, y)) + self.epsilon, np.repeat([1.0, -1.0], n), None
        if shared is not None:
            if rows is not None:
                m = shared.n
                (q, ub), active = _embed(2 * m, np.concatenate((rows, rows + m)), q, ub)
                e = np.repeat([1.0, -1.0], m)
            hessian = shared
            self.fit_times_ = {}
        elif solver_cls is SMO:
            hessian = self._smo_hessian(X, None, 'svr', X_device)
        else:
            hessian = self._build_hessian(X, None, 'svr', X_device, bias)
        solver = self._make_solver(solver_cls, hessian, q, ub, e, active)
        return dict(X=X, y=y, n=n, bias=bias, solver=solver, rows=rows)

    def _finish_fit(self, plan):
        """Everything ``fit`` does after the solver has run (ml/svm/_base.py:1275-1277, 1423-1437)."""
        X, y, n, bias = plan['X'], plan['y'], plan['n'], plan['bias']
        self.optimizer = plan['solver']
        self._after_solver(self.optimizer)
        self.alphas_ = self.optimizer.x
        alphas_p, alphas_n = np.split(self.alphas_, 2)

        # ml/svm/_base.py:1423-1437
        sv = np.logical_or(alphas_p > 1e-6, alphas_n > 1e-6)
        self.support_ = np.arange(n)[sv]
        self._set_support_vectors(X, plan['rows'])
        sv_y = y[sv]
        self.dual_coef_ = alphas_p[sv] - alphas_n[sv]
        if isinstance(self.kernel, LinearKernel):
            self.coef_ = np.dot(self.dual_coef_, self.support_vectors_)
        if isinstance(self.optimizer, SMO):
            self.intercept_ = -self.optimizer.rho
            return self
        beta = np.where(sv, alphas_p - alphas_n, 0.)
        v = self.obj.device_hessian().product(np.concatenate((beta, np.zeros(n))))[:n]  # (K + bias) beta
        k_dot = v[sv] - bias * np.sum(self.dual_coef_)
        self.intercept_ = (float(np.sum(sv_y - k_dot)) - self.epsilon) / len(sv_y)
        return self

    def predict(self, X):
        return self.decision_function(X)


class DualSVC(SVC):
    """``SVC`` preset to the path this package accelerates: hinge loss, dual problem with the intercept
    regularised, ProjectedGradient on the GPU (the name BASELINE.json uses)."""

    def __init__(self, loss=Hinge, kernel=gaussian, C=1, rho=1, mu=1, fit_intercept=True, intercept_scaling=1,
                 reg_intercept=True, dual=True, optimizer=ProjectedGradient, master_solver='clarabel',
                 learning_rate='auto', momentum_type='none', momentum=0.9, max_iter=1000, max_f_eval=15000, tol=1e-4,
                 batch_size=None, shuffle=True, random_state=None, early_stopping=False, validation_split=0.,
                 patience=5, verbose=False, master_verbose=False, shrinking=False):
        super(DualSVC, self).__init__(loss=loss, kernel=kernel, C=C, rho=rho, mu=mu, fit_intercept=fit_intercept,
                                      intercept_scaling=intercept_scaling, reg_intercept=reg_intercept, dual=dual,
                                      optimizer=optimizer, master_solver=master_solver, learning_rate=learning_rate,
                                      momentum_type=momentum_type, momentum=momentum, max_iter=max_iter,
                                      max_f_eval=max_f_eval, tol=tol, batch_size=batch_size, shuffle=shuffle,
                                      random_state=random_state, early_stopping=early_stopping,
                                      validation_split=validation_split, patience=patience, verbose=verbose,
                                      master_verbose=master_verbose, shrinking=shrinking)


class DualSVR(SVR):
    """``SVR`` preset: eps-insensitive loss, dual problem, ProjectedGradient on the GPU."""

    def __init__(self, loss=EpsilonInsensitive, epsilon=0.1, kernel=gaussian, C=1, rho=1, mu=1, fit_intercept=True,
                 intercept_scaling=1, reg_intercept=True, dual=True, optimizer=ProjectedGradient,
                 master_solver='clarabel', learning_rate='auto', momentum_type='none', momentum=0.9, max_iter=1000,
                 max_f_eval=15000, tol=1e-4, batch_size=None, shuffle=True, random_state=None, early_stopping=False,
                 validation_split=0., patience=5, verbose=False, master_verbose=False, shrinking=False):
        super(DualSVR, self).__init__(loss=loss, epsilon=epsilon, kernel=kernel, C=C, rho=rho, mu=mu,
                                      fit_intercept=fit_intercept, intercept_scaling=intercept_scaling,
                                      reg_intercept=reg_intercept, dual=dual, optimizer=optimizer,
                                      master_solver=master_solver, learning_rate=learning_rate,
                                      momentum_type=momentum_type, momentum=momentum, max_iter=max_iter,
                                      max_f_eval=max_f_eval, tol=tol, batch_size=batch_size, shuffle=shuffle,
                                      random_state=random_state, early_stopping=early_stopping,
                                      validation_split=validation_split, patience=patience, verbose=verbose,
                                      master_verbose=master_verbose, shrinking=shrinking)
