"""K11 (csrc/k_smo.cuh) on the B200: SMO fits bit-identical to oracle/smo_oracle.py on the matrix the kernel read, the
libsvm bar of tests/smo_checks.py, reproducibility, the reference's iris recipe, the KKT conditions at C4 size."""
import numpy as np
import pytest

import smo_checks as SC
from oracle import smo_oracle as SO
from optiml_b200.configs import make_config

pytestmark = pytest.mark.gpu


def fit(task, n, tol=1e-5, max_iter=10 ** 7, kernel=None, cfg=None):
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    if task == 'svc':
        spec, X, y = make_config(cfg or 'C1', n=n)
        m = SVC(loss=hinge, kernel=kernel or GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol,
                max_iter=max_iter)
    else:
        spec, X, y = make_config('C2', n=n)
        m = SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo',
                tol=tol, max_iter=max_iter)
    return m.fit(X, y), X, y


@pytest.mark.parametrize('task,kind', [('svc', 'gaussian'), ('svr', 'poly')])
def test_bit_identical_to_the_oracle_and_close_to_libsvm(task, kind):
    m, X, y = fit(task, 2000)
    o = m.optimizer
    Q = m.obj.device_hessian().to_host()
    r = SO.smo(Q, o.f.q, o.y, o.ub, tol=1e-5, max_iter=10 ** 7)
    assert o.status == r.status == 'optimal' and o.iter == r.iter
    for got, want in ((o.x, r.x), (o.g_x, r.g), (o.f_hist, r.f_hist), (o.gap_hist, r.gap_hist)):
        assert np.array_equal(got, want)
    assert o.rho == r.rho and m.intercept_ == -r.rho
    K, Qh, q, signs, C, gamma = SC.problem(task, X, y, kind)
    sk = SC.sklearn_fit(task, X, y, kind, gamma, tol=1e-5)
    SC.check_against_libsvm(task, X, K, Qh, q, signs, C, o.x, o.rho, o.gap, 1e-5, sk)


def test_two_fits_are_bitwise_equal():
    a, _, _ = fit('svc', 2000)
    b, _, _ = fit('svc', 2000)
    for u, v in ((a.optimizer.x, b.optimizer.x), (a.optimizer.g_x, b.optimizer.g_x), (a.optimizer.f_hist, b.optimizer.f_hist)):
        assert np.array_equal(u, v)
    assert a.optimizer.iter == b.optimizer.iter and a.intercept_ == b.intercept_


def test_iris_one_vs_rest(golden):
    """the reference's recipe (ml/tests/test_svc.py:96-115) with optimizer='smo'"""
    from optiml_b200.ml.multiclass import OneVsRestClassifier
    from optiml_b200.ml.svm import SVC
    from optiml_b200.ml.svm.kernels import gaussian
    from optiml_b200.ml.svm.losses import hinge
    g = golden('iris_ovr')
    ovr = OneVsRestClassifier(SVC(loss=hinge, kernel=gaussian, dual=True, optimizer='smo')).fit(g['X_train'], g['y_train'])
    assert ovr.score(g['X_test'], g['y_test']) >= 0.97
    assert all(e.optimizer.status == 'optimal' for e in ovr.estimators_)


def test_linear_kernel_coef():
    from optiml_b200.ml.svm.kernels import LinearKernel
    m, X, y = fit('svc', 1000, tol=1e-3, kernel=LinearKernel())
    assert np.allclose(m.coef_, m.dual_coef_ @ m.support_vectors_, rtol=0, atol=1e-12)
    assert np.abs(m.decision_function(X[:50]) - (X[:50] @ m.coef_ + m.intercept_)).max() <= 1e-9


def test_c4_full_size_reaches_the_kkt_conditions():
    tol = 1e-3
    m, X, y = fit('svc', None, tol=tol, cfg='C4')
    o = m.optimizer
    n, a, G, s = len(y), o.x, o.g_x, o.y
    assert o.status == 'optimal' and o.gap < tol
    assert np.all(a >= 0) and np.all(a <= 1.0)
    assert abs(s @ a) <= 1e-10 * 1.0 * n
    Qa = m.obj.device_hessian().product(a)   # one masked product
    f = 0.5 * a @ Qa - a.sum()
    assert abs(o.f_x - f) <= 1e-10 * abs(f)
    minus_yG = -s * G
    up = np.where(s > 0, a < 1.0, a > 0)
    low = np.where(s > 0, a > 0, a < 1.0)
    assert minus_yG[up].max() - minus_yG[low].min() <= tol


def test_smo_between_two_pg_fits_leaves_them_unchanged():
    from optiml_b200.ml.svm import DualSVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    spec, X, y = make_config('C1', n=1500)
    a = DualSVC(kernel=GaussianKernel(), max_iter=300).fit(X, y)
    fit('svc', 2000)
    b = DualSVC(kernel=GaussianKernel(), max_iter=300).fit(X, y)
    assert np.array_equal(a.alphas_, b.alphas_) and a.intercept_ == b.intercept_
    assert np.array_equal(np.asarray(a.train_loss_history), np.asarray(b.train_loss_history))
