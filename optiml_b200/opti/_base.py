"""Host mirror of the reference's optimisation base layer, restricted to what the dual-BCQP path
uses (reference: optiml/opti/_base.py).  Matrix work is done by the svmb200 CUDA library."""
import numpy as np

from ..runtime import DeviceHessian, GroupHessian, KernelRowsHessian, default_context, hessian_from_host


class OptimizationFunction:
    """Minimal counterpart of optiml/opti/_base.py:184-225 (no autograd: the only objective on this
    path, ``Quadratic``, has analytic derivatives)."""

    def __init__(self, ndim=2):
        self.ndim = ndim

    def x_star(self):
        return np.full(fill_value=np.nan, shape=self.ndim)

    def f_star(self):
        return np.inf

    def args(self):
        return ()

    def function(self, x):
        raise NotImplementedError

    def jacobian(self, x):
        raise NotImplementedError

    def function_jacobian(self, *args, **kwargs):
        return self.function(*args, **kwargs), self.jacobian(*args, **kwargs)

    def hessian(self, x):
        raise NotImplementedError

    def __call__(self, *args, **kwargs):
        return self.function(*args, **kwargs)


class Quadratic(OptimizationFunction):
    """f(x) = x'Qx/2 + q'x  (optiml/opti/_base.py:228-300).

    ``Q`` may be a host array (uploaded to HBM on first use, row-sharded across ranks) or a
    :class:`~optiml_b200.runtime.DeviceHessian` that already lives on the GPU(s) -- the estimators
    build it there and never hold an n x n matrix on the host.  ``.Q`` materialises a host copy on
    request only.
    """

    def __init__(self, Q, q):
        q = np.array(q, dtype=float)
        if isinstance(Q, (DeviceHessian, GroupHessian, KernelRowsHessian)):
            self._device, self._host_Q = Q, None
            n = Q.nvars
        else:
            Q = np.array(Q, dtype=float)
            n = len(Q)
            if Q.ndim != 2 or n != Q.shape[1]:
                raise ValueError('Q is not square')
            self._device, self._host_Q = None, Q
        super(Quadratic, self).__init__(n)
        if n <= 1:
            raise ValueError('Q is too small')
        if q.size != n:
            raise ValueError('q size does not match with Q')
        self.q = q

    # -- storage ------------------------------------------------------------------------------
    @property
    def Q(self):
        if self._host_Q is None:
            if self._device is None:
                raise RuntimeError('the device copy of Q was released and no host copy exists')
            self._host_Q = self._device.to_host()
        return self._host_Q

    def device_hessian(self, ctx=None):
        if self._device is None:
            if self._host_Q is None:
                raise RuntimeError('the device copy of Q was released and no host copy exists')
            self._device = hessian_from_host(ctx or default_context(), self._host_Q)
        return self._device

    def release(self):
        """Free the HBM copy of Q."""
        if self._device is not None:
            self._device.release()
            self._device = None

    def __getstate__(self):
        """Pickling / deep-copying a fitted estimator (joblib.dump, sklearn meta-estimators with n_jobs) must not
        drag device handles along: the copy keeps q and -- only if it was ever materialised -- the host Q."""
        state = self.__dict__.copy()
        state['_device'] = None
        return state

    # -- values -------------------------------------------------------------------------------
    def _Qx(self, x):
        return self.device_hessian().product(np.asarray(x, dtype=float))

    def function(self, x):
        x = np.asarray(x, dtype=float)
        return 0.5 * x @ self._Qx(x) + self.q @ x

    def jacobian(self, x):
        return self._Qx(x) + self.q

    def hessian(self, x):
        return self.Q


class Optimizer:
    """State and callback protocol shared by the solvers (optiml/opti/_base.py:9-172): plain objectives and the
    augmented-Lagrangian dual (``f.primal`` and ``f.rho`` present).  The plain Lagrangian dual of the reference
    (multipliers appended to x) is not on the path."""

    def __init__(self, f, x=None, eps=1e-6, tol=1e-8, max_iter=1000, callback=None, callback_args=(),
                 random_state=None, verbose=False):
        if not isinstance(f, OptimizationFunction):
            raise TypeError(f'{f} is not an allowed optimization function')
        self.f = f
        if x is None:
            x = (np.random.uniform if random_state is None else np.random.RandomState(random_state).uniform)
        self.x = x(size=f.ndim) if callable(x) else np.asarray(x, dtype=float)
        self.f_x = np.nan
        if self.is_lagrangian_dual():  # optiml/opti/_base.py:66-69
            self.past_x = self.x.copy()
            self.primal_f_x = np.nan
            self.dgap = np.nan
        self.g_x = np.zeros(0)
        self.eps = eps
        self.tol = tol
        if not max_iter > 0:
            raise ValueError('max_iter must be > 0')
        self.max_iter = max_iter
        self.iter = 0
        self.status = 'unknown'
        if self.f.ndim <= 3 or (hasattr(self.f, 'primal') and self.f.primal.ndim <= 3):
            self.x0_history, self.x1_history, self.f_x_history = [], [], []
        self._callback = callback
        self.callback_args = callback_args
        self.random_state = random_state
        self.verbose = verbose

    def is_lagrangian_dual(self):
        return hasattr(self.f, 'primal')

    def is_augmented_lagrangian_dual(self):
        return self.is_lagrangian_dual() and hasattr(self.f, 'rho')

    def callback(self, args=()):
        if self.is_lagrangian_dual():
            # optiml/opti/_base.py:96-117; primal_f_x (= primal.function(x)) is set by the device loop, which gets
            # x'Qx from the same streaming pass that produced the gradient
            self.dgap = abs((self.primal_f_x - self.f_x) / max(abs(self.primal_f_x), 1))
            if self.is_verbose():
                print('\tpcost: {: 1.4e}'.format(self.primal_f_x), end='')
                print('\tdgap: {: 1.4e}'.format(self.dgap), end='')
            if self.f.primal.ndim == 2:
                self.x0_history.append(self.x[0])
                self.x1_history.append(self.x[1])
                self.f_x_history.append(self.primal_f_x)
            if callable(self._callback):
                self._callback(self, *args, *self.callback_args)
            self.past_x = self.x.copy()
            return
        if self.f.ndim <= 3:
            self.x0_history.append(self.x[0])
            self.x1_history.append(self.x[1])
            self.f_x_history.append(self.f_x)
        if callable(self._callback):
            self._callback(self, *args, *self.callback_args)

    def is_verbose(self):
        return self.verbose and not self.iter % self.verbose

    def minimize(self):
        raise NotImplementedError
