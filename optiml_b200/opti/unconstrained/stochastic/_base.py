"""Full-batch stochastic optimisers on the augmented-Lagrangian dual, run on the GPU(s).

Host mirror of optiml/opti/unconstrained/stochastic/_base.py:13-140 (constructors, validation, attributes, verbose
output) for the one use the SVM dual path makes of them (ml/svm/_base.py:638-725, 1188-1270): ``f`` is an
``AugmentedLagrangianQuadratic`` and every iteration sees the whole problem (``batch_size=None``).  The loop --
value and gradient of the Lagrangian, update rule, multiplier update, optimality test -- is ``svmb200_al_*``
(csrc/pg.cu, csrc/k3_vector.cuh, csrc/al_math.cuh): one streaming pass over Q and one vector kernel per iteration.
"""
import ctypes as C
import itertools
from collections.abc import Iterable

import numpy as np

from .schedules import constant
from ... import Optimizer
from ...constrained import AugmentedLagrangianQuadratic
from ...constrained._device_loop import DeviceLoopMixin, create_solvers, destroy_solvers
from .... import _native as N


class _StepSize:
    """``step_size(*batch)`` -> iterator, the protocol of stochastic/_base.py:82-87 -- as a picklable object (the
    reference wraps scalars and iterables in lambdas, which makes its fitted estimators unpicklable)."""

    def __init__(self, value, is_iterable):
        self.value, self.is_iterable = value, is_iterable

    def __call__(self, *args):
        return self.value if self.is_iterable else constant(self.value)


class StochasticOptimizer(DeviceLoopMixin, Optimizer):
    _rule = None            # name of the update rule in _native.RULES
    _momentum_capable = False

    def __init__(self, f, x=None, step_size=0.01, batch_size=None, eps=1e-6, tol=1e-8, epochs=1000, callback=None,
                 callback_args=(), shuffle=True, random_state=None, verbose=False):
        super(StochasticOptimizer, self).__init__(f=f, x=x, eps=eps, tol=tol, max_iter=epochs, callback=callback,
                                                  callback_args=callback_args, random_state=random_state,
                                                  verbose=verbose)
        if not callable(step_size) and not isinstance(step_size, Iterable) and not step_size > 0:
            raise ValueError('step_size must be > 0 or a callable or an iterator')
        if isinstance(step_size, Iterable):
            self.step_size = _StepSize(step_size, True)
        elif callable(step_size):
            self.step_size = step_size
        else:
            self.step_size = _StepSize(step_size, False)
        self.epochs = epochs
        self.epoch = 0
        self.shuffle = shuffle
        self.step = 0
        if batch_size is not None:
            raise NotImplementedError('mini batches do not apply to the augmented-Lagrangian dual (f.args() is empty)')
        self.batch_size = None
        self.batches = itertools.repeat(f.args())

    def is_batch_end(self):
        return True

    def is_verbose(self):
        return self.verbose and not self.epoch % self.verbose

    # ------------------------------------------------------------------ rule constants
    def _rule_constants(self):
        """decay, beta1, beta2, offset for svmb200_al_create (unused ones keep their neutral defaults)"""
        return dict(decay=getattr(self, 'decay', 0.9), beta1=getattr(self, 'beta1', 0.9),
                    beta2=getattr(self, 'beta2', 0.999), offset=getattr(self, 'offset', 1e-8))

    def _draw(self, source, count):
        """the first ``count`` values of a schedule (an iterator, or an iterable re-read from its start)"""
        vals = np.fromiter(itertools.islice(iter(source), count), dtype=np.float64)
        if len(vals) < count:
            raise ValueError(f'schedule ended after {len(vals)} values, {count} are needed')
        return vals

    # ------------------------------------------------------------------ device solver handle
    def _create(self, profile=False):
        f = self.f
        if not isinstance(f, AugmentedLagrangianQuadratic):
            raise NotImplementedError('the device loop drives AugmentedLagrangianQuadratic objectives only')
        H = f.device_hessian()
        n = H.nvars
        if self.x.size != n:
            raise ValueError('start point size does not match with Q')
        if self.random_state is None:
            # an unseeded start point (opti/_base.py:40-41) differs from rank to rank: all ranks take rank 0's
            # (under torchrun; the ranks of a single-process group are created from this one array anyway)
            if getattr(H, 'group', None) is None:
                self.x = H.ctx.broadcast_array(self.x)
        q, lb, ub, x0 = (np.ascontiguousarray(v, dtype=np.float64) for v in (f.q, f.lb, f.ub, self.x))
        a = np.ascontiguousarray(f.A[0]) if f.n_eq else None
        b = float(f.b[0]) if f.n_eq else 0.
        lr = self._draw(self.step_size(*f.args()), self.epochs)
        momentum_type = getattr(self, 'momentum_type', 'none')
        mom = self._draw(self.momentum, self.epochs + 1) if momentum_type != 'none' else None
        k = self._rule_constants()
        h = create_solvers('svmb200_al_create', H, lambda hh: (
            N.ptr(q), N.ptr(lb), N.ptr(ub), N.ptr(x0), N.ptr(a), b, float(f.rho), N.RULES[self._rule],
            N.MOMENTUM[momentum_type], N.ptr(lr), N.ptr(mom), float(k['decay']), float(k['beta1']), float(k['beta2']),
            float(k['offset']), float(self.tol), int(self.epochs), C.byref(hh)))
        self._after_create(h, profile)
        return h, n

    def _pull_state(self, h, n):
        self.primal_f_x = super(StochasticOptimizer, self)._pull_state(h, n)  # second scalar = primal cost
        return self.primal_f_x

    def _pull_multipliers(self, h, n):
        f = self.f
        mu = C.c_double(0)
        lam_lb, lam_ub = np.empty(n), np.empty(n)
        N.call('svmb200_al_multipliers', h, C.byref(mu), N.ptr(lam_lb), N.ptr(lam_ub))
        f.dual_x = np.concatenate(([mu.value] if f.n_eq else [], lam_lb, lam_ub))

    def _print_header(self):
        if self.verbose:
            print('epoch\titer\t cost\t', end='')  # _base.py:121-123 (f_star() is inf here: no gap / rate columns)

    def _print_info(self):
        if self.is_verbose():
            print('\n{:4d}\t{:4d}\t{: 1.4e}'.format(self.epoch, self.iter, self.f_x), end='')  # _base.py:128-130

    def _problem_ndim(self):
        return self.f.primal.ndim

    def minimize(self):
        self._print_header()
        h, n = self._create(bool(getattr(self, 'profile', False)))
        try:
            if self._resident_ok():
                self._minimize_resident(h, n)
            else:
                self._minimize_stepwise(h, n)
            self._after_run(h, n)
        finally:
            destroy_solvers(h)
        if self.verbose:
            print('\n')
        return self

    def _after_run(self, h, n):
        self._pull_multipliers(h, n)
        self._collect_stats(h)
        assert all(self.f.dual_x[self.f.n_eq:] >= 0)  # opti/_base.py:163-167

    def _finish_resident(self, h, n, it, status):
        # whole loop on the device; L and the primal cost at every callback point come back in one copy
        self.iter, self.status = it, status
        self._pull_state(h, n)
        self.epoch = self.iter + 1
        cnt = C.c_int64(0)
        f_hist, pf_hist = np.empty(self.iter + 1), np.empty(self.iter + 1)
        N.call('svmb200_pg_history', h, N.ptr(f_hist), N.ptr(pf_hist), C.byref(cnt))
        self.f_hist, self.pf_hist = f_hist[:cnt.value], pf_hist[:cnt.value]
        self.dgap = abs((self.primal_f_x - self.f_x) / max(abs(self.primal_f_x), 1))
        if self._callback is not None and not self._extend_owner_history(self.pf_hist):   # the primal cost (ml/svm/_base.py:291)
            final = (self.iter, self.f_x, self.primal_f_x)
            for k, (fk, pk) in enumerate(zip(self.f_hist, self.pf_hist)):
                self.iter, self.f_x, self.primal_f_x = k, float(fk), float(pk)
                self._callback(self, *self.callback_args)
            self.iter, self.f_x, self.primal_f_x = final

    def _minimize_stepwise(self, h, n):
        # generic callbacks / verbose / tiny problems: synchronise at every callback point (adagrad.py:88-121)
        self.iter, status = self._run(h, 0)
        while True:
            self._pull_state(h, n)
            self._print_info()
            try:
                self.callback()
            except StopIteration:
                break
            self.epoch += 1
            if status == 'stopped':          # epoch limit reached at this state
                self.status = status
                break
            self.iter, status = self._run(h, 1)
            if status == 'optimal':          # the multiplier update of this iteration met the optimality test:
                self.status = status         # x moved, f_x / g_x stay those of the last evaluation
                x = np.empty(n)
                N.call('svmb200_pg_state', h, N.ptr(x), None, None, None)
                self.x = x
                break


class StochasticMomentumOptimizer(StochasticOptimizer):
    _momentum_capable = True

    def __init__(self, f, x=None, step_size=0.01, momentum_type='none', momentum=0.9, batch_size=None, eps=1e-6,
                 tol=1e-8, epochs=1000, callback=None, callback_args=(), shuffle=True, random_state=None,
                 verbose=False):
        super(StochasticMomentumOptimizer, self).__init__(f=f, x=x, step_size=step_size, batch_size=batch_size,
                                                          eps=eps, tol=tol, epochs=epochs, callback=callback,
                                                          callback_args=callback_args, shuffle=shuffle,
                                                          random_state=random_state, verbose=verbose)
        if momentum_type not in ('polyak', 'nesterov', 'none'):
            raise ValueError(f'unknown momentum type {momentum_type}')
        self.momentum_type = momentum_type
        if not isinstance(momentum, Iterable) and not 0 <= momentum < 1:
            raise ValueError('momentum must be between 0 and 1 or an iterator')
        self.momentum = momentum if isinstance(momentum, Iterable) else constant(momentum)
