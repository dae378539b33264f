"""Shared checks of the SMO solver (csrc/k_smo.cuh, oracle/smo_oracle.py) against libsvm through ``sklearn.svm``.

libsvm solves the same problem (it is the algorithm's origin) but caches kernel rows in FP32 and shrinks, so the two
trajectories differ; the solutions agree to the solver tolerance.  The bars below were calibrated on the CPU at
tol = 1e-5: on the cases of tests/test_smo_oracle.py the objectives agree to 1e-11 relative, the decision values to
1.4e-4 (the linear case; 2e-5 otherwise), the intercepts to 1e-5.
"""
import numpy as np

from oracle import svm_oracle as O
from oracle import smo_oracle as SO

SK_KERNEL = {'gaussian': 'rbf', 'poly': 'poly', 'linear': 'linear'}


def problem(task, X, y, kind, C=1., epsilon=0.1, degree=3, coef0=0.):
    """(K, Q, q, signs, C vector, gamma) of the dual as the estimators pose it with reg_intercept=False."""
    gamma = O.resolve_gamma('scale', X)
    K = O.kernel_matrix(kind, X, None, degree=degree, gamma=gamma, coef0=coef0)
    n = len(y)
    if task == 'svc':
        ys = np.where(y == np.unique(y)[1], 1., -1.)
        return K, ys[:, None] * K * ys[None, :], -np.ones(n), ys, np.full(n, float(C)), gamma
    y = np.asarray(y, dtype=float)
    return K, SO.full_q(K, 'svr'), np.hstack((-y, y)) + epsilon, np.hstack((np.ones(n), -np.ones(n))), \
        np.full(2 * n, float(C)), gamma


def sklearn_fit(task, X, y, kind, gamma, C=1., tol=1e-5, epsilon=0.1, degree=3, coef0=0.):
    from sklearn.svm import SVC, SVR
    kw = dict(kernel=SK_KERNEL[kind], C=C, tol=tol, gamma=gamma, degree=degree, coef0=coef0, cache_size=2000)
    return (SVC(**kw) if task == 'svc' else SVR(epsilon=epsilon, **kw)).fit(X, y)


def sklearn_alpha(task, sk, n):
    """libsvm's dual variables in the layout of our problem (SVC: n alphas; SVR: [alpha+, alpha-])."""
    coef = np.zeros(n)
    coef[sk.support_] = sk.dual_coef_.ravel()
    if task == 'svc':
        return np.abs(coef)
    return np.hstack((np.maximum(coef, 0.), np.maximum(-coef, 0.)))


def check_against_libsvm(task, X, K, Q, q, signs, C, alpha, rho, gap, tol, sk):
    """The libsvm bar of the SMO tests: alpha, rho and exit gap of our solve against the sklearn model ``sk`` fitted on
    the same data, both dual objectives evaluated in FP64 on the same Q."""
    n = K.shape[0]
    a_sk = sklearn_alpha(task, sk, n)
    f = 0.5 * alpha @ (Q @ alpha) + q @ alpha
    f_sk = 0.5 * a_sk @ (Q @ a_sk) + q @ a_sk
    assert abs(f - f_sk) <= 1e-6 * abs(f_sk), (f, f_sk)
    coef = signs * alpha if task == 'svc' else alpha[:n] - alpha[n:]
    dec, dec_sk = K @ coef - rho, (sk.decision_function(X) if task == 'svc' else sk.predict(X))
    assert np.abs(dec - dec_sk).max() <= 1e-3, np.abs(dec - dec_sk).max()
    if task == 'svc':
        sure = np.abs(dec_sk) > 1e-3
        assert np.array_equal(dec[sure] > 0, dec_sk[sure] > 0)
    near_bound = (np.minimum(alpha, C - alpha) < 1e-4 * C) | (np.minimum(a_sk, C - a_sk) < 1e-4 * C)
    assert np.array_equal((alpha > 0)[~near_bound], (a_sk > 0)[~near_bound])
    assert abs(-rho - float(np.ravel(sk.intercept_)[0])) <= 1e-3
    assert gap < tol
    assert abs(signs @ alpha) <= 1e-12 * C.max() * len(alpha)
    return f, f_sk
