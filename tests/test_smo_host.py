"""Host logic of optimizer='smo': estimator dispatch, scope guards, sklearn protocol, the C ABI's refusals."""
import ctypes as C

import numpy as np
import pytest
from sklearn.base import clone

from emu import emulated_device
from optiml_b200 import _native as N
from optiml_b200.configs import make_config
from optiml_b200.ml.svm import SVC, SVR
from optiml_b200.ml.svm.kernels import GaussianKernel
from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
from optiml_b200.ml.svm.smo import SMO
from optiml_b200.opti.constrained import ProjectedGradient


def svc(**kw):
    return SVC(loss=hinge, kernel=GaussianKernel(), dual=True, optimizer='smo', tol=1e-5, **kw)


def test_dispatch():
    assert svc()._bcqp_solver_class() is SMO
    assert SVR(loss=epsilon_insensitive, dual=True, optimizer='smo')._bcqp_solver_class() is SMO
    with pytest.raises(NotImplementedError, match='ProjectedGradient or FrankWolfe'):
        svc(reg_intercept=True)._bcqp_solver_class()
    with pytest.raises(NotImplementedError):
        SVC(loss=hinge, dual=True, optimizer='cvxopt')._bcqp_solver_class()
    with pytest.raises(NotImplementedError):   # the BCQP solvers keep needing reg_intercept=True
        SVC(loss=hinge, dual=True, optimizer=ProjectedGradient)._bcqp_solver_class()
    assert not hasattr(svc(), 'train_loss_history')   # string optimizers keep no history on the estimator


def test_sharded_fit_is_refused_before_any_device_work(monkeypatch):
    from optiml_b200 import runtime

    class ShardedContext:   # what default_context() is under torchrun with two ranks; any device call would fail
        nranks, group = 2, None
    monkeypatch.setattr(runtime, '_default_ctx', ShardedContext())
    spec, X, y = make_config('C1', n=64)
    with pytest.raises(NotImplementedError, match='one GPU'):
        svc().fit(X, y)
    with pytest.raises(NotImplementedError, match='one GPU'):
        SVR(loss=epsilon_insensitive, dual=True, optimizer='smo').fit(X, y.astype(float))


def test_clone_params_refit_and_no_lockstep():
    from optiml_b200.ml.multiclass import _lockstep_capable
    m = svc(C=2)
    assert m.get_params()['optimizer'] == 'smo' and clone(m).get_params()['optimizer'] == 'smo'
    assert not _lockstep_capable(m)
    spec, X, y = make_config('C1', n=90)
    with emulated_device():
        m.fit(X, y)
        first = m.optimizer
        assert isinstance(first, SMO) and first.status == 'optimal'
        assert not _lockstep_capable(m)
        m.fit(X, y)   # refit: the fitted SMO instance stands for 'smo'
        assert m.optimizer is not first and np.array_equal(m.optimizer.x, first.x)
        assert clone(svc(C=2)).fit(X, y).intercept_ == m.intercept_


def test_abi_refuses_a_partial_shard():
    from optiml_b200.runtime import DeviceHessian, default_context
    n = 40
    y, q, ub = np.ones(n), -np.ones(n), np.ones(n)
    with emulated_device() as lib:
        ctx = default_context()
        H = DeviceHessian(ctx, n)
        h = C.c_void_p()
        for row0, nrows in ((0, n - 8), (8, n - 8)):
            rc = lib.svmb200_smo_create(ctx.handle, C.c_void_p(H.matrix.dptr), n, H.ld, row0, nrows, N.HESSIAN_PLAIN,
                                        N.ptr(y), N.ptr(q), N.ptr(ub), 1e-3, 100, C.byref(h))
            assert rc == 1 and not h.value   # SVMB200_ERR_ARG
            assert b'whole matrix' in lib.svmb200_last_error()
        H.release()
