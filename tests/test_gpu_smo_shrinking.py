"""Shrinking in K11 / K12 / K14 on the B200: fits with ``shrinking=True`` bit-identical to tests/smo_shrinking_oracle.py
on the matrix the kernel read (resident and computed rows), C4 and the n = 200 000 computed fit at the KKT conditions
recomputed through K6, and the shared one-vs-rest / grid-search paths equal to sklearn's clone path."""
import numpy as np
import pytest

import smo_batch_checks as SB
import smo_cv_checks as CV
import smo_shrinking_oracle as SSO
from optiml_b200.configs import make_config

pytestmark = pytest.mark.gpu


def fit(task, n, tol=1e-5, max_iter=10 ** 7, cfg=None, shrinking=True):
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    if task == 'svc':
        spec, X, y = make_config(cfg or 'C1', n=n)
        m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=max_iter,
                shrinking=shrinking)
    else:
        spec, X, y = make_config('C2', n=n)
        m = SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo',
                tol=tol, max_iter=max_iter, shrinking=shrinking)
    return m.fit(X, y), X, y


def kkt_gap_from_k6(m):
    """m - M of the fit's alpha with G = Q alpha + q from one masked product (K6), independent of the solver's G"""
    o = m.optimizer
    a, ys = o.x, o.y
    G = m.obj.device_hessian().product(a) + o.f.q
    np.testing.assert_allclose(G, o.g_x, rtol=0, atol=1e-8 * max(1.0, np.abs(o.g_x).max()))
    up = np.where(ys > 0, a < o.ub, a > 0)
    low = np.where(ys > 0, a > 0, a < o.ub)
    return np.max(-(ys * G)[up]) - np.min(-(ys * G)[low])


@pytest.mark.parametrize('rows', ['resident', 'computed'])
@pytest.mark.parametrize('task', ['svc', 'svr'])
def test_bit_identical_to_the_oracle(monkeypatch, task, rows):
    monkeypatch.setenv('SVMB200_SMO_ROWS', rows)
    m, X, y = fit(task, 2000)
    o = m.optimizer
    assert o.row_source == rows
    Q = m.obj.device_hessian().to_host()
    r = SSO.smo(Q, o.f.q, o.y, o.ub, tol=1e-5, max_iter=10 ** 7, shrinking=True)
    assert o.status == r.status == 'optimal' and o.iter == r.iter and r.checks >= 1
    for got, want in ((o.x, r.x), (o.g_x, r.g), (o.f_hist, r.f_hist), (o.gap_hist, r.gap_hist)):
        assert np.array_equal(got, want)
    assert o.rho == r.rho and m.intercept_ == -r.rho
    assert (o.active_, o.shrink_checks, o.reconstructions) == (r.active, r.checks, r.reconstructions)


def test_c4_full_size_reaches_the_kkt_conditions():
    tol = 1e-3
    m, X, y = fit('svc', None, tol=tol, cfg='C4')
    o = m.optimizer
    assert o.status == 'optimal' and o.gap < tol and o.shrink_checks >= 1 and o.active_ < len(y)
    assert kkt_gap_from_k6(m) <= tol
    plain, _, _ = fit('svc', None, tol=tol, cfg='C4', shrinking=False)
    assert abs(o.f_x - plain.optimizer.f_x) <= 1e-4 * abs(plain.optimizer.f_x)
    print(f'C4: {o.iter} iterations with shrinking ({plain.optimizer.iter} without), {o.active_} active at the last '
          f'check, {o.shrink_checks} checks, {o.reconstructions} reconstructions')


def test_one_vs_rest_equals_clone_per_class():
    spec, X, _ = make_config('C1')
    y = SB.quantile_classes(X, 4)
    ours, theirs = SB.compare_ovr(SB.svc(tol=1e-3, max_iter=10 ** 6, shrinking=True), X, y)
    SB.assert_one_shared_matrix(ours.estimators_)


def test_grid_search_over_shrinking_equals_sklearns():
    spec, X, _ = make_config('C1')
    y = (SB.quantile_classes(X, 10) == 0).astype(int)
    CV.grid_search_both(SB.svc(tol=1e-3, max_iter=10 ** 6), {'C': [0.3, 1.0, 3.0], 'shrinking': [False, True]}, X, y,
                        cv=5)


def test_large_computed_fit_reaches_the_kkt_conditions(monkeypatch):
    monkeypatch.delenv('SVMB200_SMO_ROWS', raising=False)
    monkeypatch.delenv('SVMB200_SMO_CACHE_MB', raising=False)
    n, tol = 200_000, 1e-3
    from optiml_b200.ml.svm import SVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge
    spec, X, y = make_config('C5', n=n)
    m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=10 ** 7,
            shrinking=True).fit(X, y)
    o = m.optimizer
    assert o.row_source == 'computed' and o.status == 'optimal' and o.gap < tol
    gap = kkt_gap_from_k6(m)
    assert gap <= tol
    print(f'n = {n}: {o.iter} iterations, {o.device_ms / 1e3:.2f} s solve, {o.active_} active at the last check, '
          f'{o.reconstructions} reconstructions, KKT gap from K6 {gap:.3e}')
    m.obj.release()
