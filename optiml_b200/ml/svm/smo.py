"""Sequential minimal optimization for the SVM dual with its equality constraint, run on the GPU.

Where the reference keeps its SMO (optiml/ml/svm/smo.py: SMOClassifier, SMORegression) this module keeps the host mirror
of K11 (csrc/k_smo.cuh): libsvm's solver without shrinking (Fan, Chen & Lin 2005, working-set selection WSS2) for

    min a'Qa/2 + q'a   s.t.  y'a = 0,  0 <= a <= C

-- the problem ``sklearn.svm.SVC`` / ``SVR`` solve, i.e. an unregularised intercept.  The reference's own selection rules
(Platt / Keerthi) are not reproduced: the algorithm is the one csrc/k_smo.cuh documents.  The estimators reach it with
``optimizer='smo'`` (and ``reg_intercept=False``).
"""
import ctypes as C
import os

import numpy as np

from ... import _native as N
from ...opti import Optimizer, Quadratic
from ...opti.constrained._device_loop import DeviceLoopMixin
from ...runtime import KernelRowsHessian

RESIDENT_SHARE = 0.9   # the resident matrix may take this share of the free device memory
CACHE_SHARE = 0.8      # the row cache of the computed form may take this share of what is free once X is in place


def select_row_source(n, nvars, ld, d, info):
    """Where an SMO fit of ``n`` samples (``nvars`` variables, ``d`` features) gets the rows of Q: ``('resident', 0)``
    when the n x ld matrix fits ``RESIDENT_SHARE`` of ``info['free_bytes']`` (``Context.info()`` after ``trim()``), else
    ``('computed', cache_bytes)`` with a row cache of ``CACHE_SHARE`` of what X leaves free, at most all n rows.  Raises
    ``ValueError`` before any device work when the computed form cannot hold ``nvars`` (the shared-memory slice:
    ``svmb200_smo_max_vars``).  ``SVMB200_SMO_ROWS=resident|computed`` and ``SVMB200_SMO_CACHE_MB`` override the
    choice and the cache size (tests, sweeps)."""
    free = int(info['free_bytes'])
    source = 'resident' if n * ld * 8 <= RESIDENT_SHARE * free else 'computed'
    forced = os.environ.get('SVMB200_SMO_ROWS', '').strip().lower()
    if forced:
        if forced not in ('resident', 'computed'):
            raise ValueError(f'SVMB200_SMO_ROWS must be resident or computed, not {forced!r}')
        source = forced
    if source == 'resident':
        return source, 0
    cap = int(N.load_library().svmb200_smo_max_vars(int(info['sm_count'])))
    if nvars > cap:
        raise ValueError(f"optimizer='smo' holds at most {cap} variables on this GPU ({cap // max(int(info['sm_count']), 1)} "
                         f"per SM, the shared-memory slice); this fit has {nvars}")
    row = nvars * 8
    mb = os.environ.get('SVMB200_SMO_CACHE_MB', '').strip()
    if mb:
        cache = int(float(mb) * (1 << 20))
    else:
        cache = int(CACHE_SHARE * max(free - n * (d + (d & 1)) * 8, 0))   # the fit's copy of X, ld = d rounded to even
    return source, min(cache // row, n) * row


def calculate_rho(alpha, G, y, C):
    """libsvm's Solver::calculate_rho: the mean of y_t G_t over the free variables (0 < alpha_t < C_t); without any, the
    middle of the interval the KKT conditions leave.  The decision function's intercept is -rho."""
    yG = y * G
    free = (alpha > 0) & (alpha < C)
    if np.any(free):
        return float(np.sum(yG[free]) / np.count_nonzero(free))
    at_lo, at_hi = alpha <= 0, alpha >= C
    ub_set = ((y > 0) & at_lo) | ((y < 0) & at_hi)
    lb_set = ((y > 0) & at_hi) | ((y < 0) & at_lo)
    ub = np.min(yG[ub_set]) if np.any(ub_set) else np.inf
    lb = np.max(yG[lb_set]) if np.any(lb_set) else -np.inf
    return float((ub + lb) / 2)


class SMO(DeviceLoopMixin, Optimizer):
    """``min x'Qx/2 + q'x : y'x = 0, 0 <= x <= C`` by SMO on the resident Hessian of ``quad`` (the whole matrix on one GPU).

    ``y``: the sign row of the equality constraint (+-1: the labels for SVC, ``[1, ..., -1, ...]`` for SVR); ``C``: the
    upper bounds (a scalar or one per variable); ``tol``: stop when the maximal violating pair's gap m - M drops below it.
    After ``minimize``: ``x`` (alpha), ``g_x`` (G = Qx + q), ``f_x`` (= sum x_t (G_t + q_t) / 2), ``iter``, ``status``
    ('optimal' or 'stopped'), ``gap``, ``f_hist`` / ``gap_hist`` (one entry per evaluated state 0 .. iter) and ``rho``
    (libsvm's; the intercept is -rho).

    ``active`` (one bool per variable, on a shared signed view only): solve the problem on the active variables alone,
    every other one held at 0 (``svmb200_smo_create_subset``) -- a cross-validation fold on the matrix of a larger set of
    rows.  ``x``, ``g_x``, ``f_x`` and ``rho`` then describe the active variables only, compacted in index order, and
    ``f_x`` and ``rho`` come from the compacted arrays, exactly as a solve of the fold's own problem computes them.

    ``shrinking``: libsvm's shrinking heuristic (``svmb200_smo_set_shrinking``): every min(l, 1000) states the variables
    at a bound that cannot enter the maximal violating pair are set aside, and their G is rebuilt before the solver
    stops.  It follows its own trajectory (csrc/k_smo.cuh).  After a run: ``active_`` (active variables after the last
    shrink check), ``shrink_checks`` and ``reconstructions``."""

    _verbose_header = 'iter\t cost\t\t gap'

    def __init__(self, quad, y, C, tol=1e-3, max_iter=1000, callback=None, callback_args=(), verbose=False, active=None,
                 shrinking=False):
        if not isinstance(quad, Quadratic):
            raise TypeError(f'{quad} is not an allowed quadratic function')
        n = quad.ndim
        y = np.asarray(y, dtype=float).ravel()
        if y.size != n or not np.all(np.abs(y) == 1):
            raise ValueError('y must hold one sign (+-1) per variable')
        C = np.broadcast_to(np.asarray(C, dtype=float), (n,)).copy()
        if not np.all(C > 0):
            raise ValueError('C must be > 0')
        if not tol >= 0:
            raise ValueError('tol must be >= 0')
        super(SMO, self).__init__(f=quad, x=np.zeros(n), eps=tol, tol=tol, max_iter=max_iter, callback=callback,
                                  callback_args=callback_args, verbose=verbose)
        if active is not None:
            active = np.asarray(active, dtype=bool).ravel()
            if active.size != n:
                raise ValueError('active must hold one flag per variable')
        self.y, self.ub, self.active, self.shrinking = y, C, active, bool(shrinking)
        self.active_, self.shrink_checks, self.reconstructions = n, 0, 0
        self.gap, self.rho = np.nan, np.nan
        self.row_source, self.cache_slots, self.cache_hits, self.cache_misses = None, 0, 0, 0

    def _create(self, profile=False):
        h, n = self._create_solver()
        if self.shrinking:
            try:
                N.call('svmb200_smo_set_shrinking', h, 1)
            except Exception:
                N.load_library().svmb200_pg_destroy(h)
                raise
        return h, n

    def _create_solver(self):
        H = self.f.device_hessian()
        q, y, ub = (np.ascontiguousarray(v, dtype=np.float64) for v in (self.f.q, self.y, self.ub))
        self.symmetric_pass = False
        if self.active is not None and (isinstance(H, KernelRowsHessian) or (H.signs is None and H.layout != 'svr')):
            raise ValueError('an active subset needs a shared resident matrix read as a signed view')
        if isinstance(H, KernelRowsHessian):
            layout = N.HESSIAN_SVR if H.layout == 'svr' else N.HESSIAN_PLAIN
            if not np.array_equal(y, H.row_signs):
                raise ValueError('with computed rows the sign row y must be the signs of the Hessian')
            h = C.c_void_p()
            N.call('svmb200_smo_create_rows', H.ctx.handle, C.c_void_p(H.X.dptr), H.n, H.X.ld, H.X.cols, int(H.kernel),
                   float(H.gamma), float(H.coef0), float(H.degree), layout, N.ptr(y), N.ptr(q), N.ptr(ub),
                   float(self.tol), int(self.max_iter), H.cache_bytes, C.byref(h))
            self.row_source = 'computed'
            return h, H.nvars
        if len(H.shards()) != 1 or H.nrows != H.n:
            raise NotImplementedError('SMO runs on one GPU: the Hessian must not be sharded')
        n = H.nvars
        layout = N.HESSIAN_SVR if H.layout == 'svr' else N.HESSIAN_PLAIN
        symbol = 'svmb200_smo_create'
        if H.signs is not None:
            # Q = (s s') o M on a shared, unsigned M (one-vs-rest, ml/multiclass.py): the kernel signs what it reads
            if not np.array_equal(y, H.signs):
                raise ValueError('on a signed view the sign row y must be the signs of the view')
            symbol = 'svmb200_smo_create_signed'
        h = C.c_void_p()
        if self.active is not None:
            # the SVR view reads M with the signs e, which is the plain SVR read (svmb200_smo_create_signed)
            if H.layout == 'svr' and not np.array_equal(y, np.repeat([1.0, -1.0], H.n)):
                raise ValueError('on an SVR matrix the sign row y must be e = [1, ..., -1, ...]')
            active = np.ascontiguousarray(self.active, dtype=np.uint8)
            N.call('svmb200_smo_create_subset', H.ctx.handle, C.c_void_p(H.matrix.dptr), H.n, H.ld, H.row0, H.nrows,
                   layout, N.ptr(y), N.ptr(q), N.ptr(ub), active.ctypes.data_as(C.c_void_p), float(self.tol),
                   int(self.max_iter), C.byref(h))
        else:
            N.call(symbol, H.ctx.handle, C.c_void_p(H.matrix.dptr), H.n, H.ld, H.row0, H.nrows, layout,
                   N.ptr(y), N.ptr(q), N.ptr(ub), float(self.tol), int(self.max_iter), C.byref(h))
        self.row_source = 'resident'
        return h, n

    def _print_iteration(self, scalars):
        print('\n{:4d}\t{: 1.4e}\t{: 1.4e}'.format(self.iter, self.f_x, scalars[1]), end='')

    def _after_run(self, h, n):
        self._collect_stats(h)
        slots, hits, misses = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        N.call('svmb200_smo_cache_stats', h, None, C.byref(slots), C.byref(hits), C.byref(misses))
        self.cache_slots, self.cache_hits, self.cache_misses = slots.value, hits.value, misses.value
        active, checks, recons = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        N.call('svmb200_smo_shrink_stats', h, C.byref(active), C.byref(checks), C.byref(recons))
        self.active_, self.shrink_checks, self.reconstructions = active.value, checks.value, recons.value
        self.gap = self._pull_state(h, n)
        cnt = C.c_int64(0)
        f_hist, gap_hist = np.empty(self.iter + 1), np.empty(self.iter + 1)
        N.call('svmb200_pg_history', h, N.ptr(f_hist), N.ptr(gap_hist), C.byref(cnt))
        self.f_hist, self.gap_hist = f_hist[:cnt.value], gap_hist[:cnt.value]
        q, y, ub = self.f.q, self.y, self.ub
        if self.active is not None:
            # zeros in a longer vector would change np.dot's rounding, and the held variables would enter rho's ub_set
            keep = self.active
            self.x, self.g_x, q, y, ub = self.x[keep], self.g_x[keep], q[keep], y[keep], ub[keep]
        self.f_x = float(0.5 * np.dot(self.x, self.g_x + q))
        self.rho = calculate_rho(self.x, self.g_x, y, ub)
