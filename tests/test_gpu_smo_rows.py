"""K12 (SMO with computed rows) on the B200: kernel rows against K1, fits bit-identical to oracle/smo_oracle.py on the
matrix assembled from svmb200_kernel_rows and within the libsvm bar of tests/smo_checks.py, cache size without effect on
the bits, a 200 000-sample fit whose 320 GB Hessian does not fit in HBM, and the other solvers unchanged around it."""
import ctypes as C

import numpy as np
import pytest

import smo_checks as SC
from oracle import smo_oracle as SO
from optiml_b200.configs import make_config

pytestmark = pytest.mark.gpu


def fit(monkeypatch, task, n, rows, cache_mb=None, tol=1e-5, cfg='C1'):
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    monkeypatch.setenv('SVMB200_SMO_ROWS', rows)
    if cache_mb is None:
        monkeypatch.delenv('SVMB200_SMO_CACHE_MB', raising=False)
    else:
        monkeypatch.setenv('SVMB200_SMO_CACHE_MB', str(cache_mb))
    if task == 'svc':
        spec, X, y = make_config(cfg, n=n)
        m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=10 ** 7)
    else:
        spec, X, y = make_config('C2', n=n)
        m = SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo',
                tol=tol, max_iter=10 ** 7)
    return m.fit(X, y), X, y


KID = {'linear': 0, 'poly': 1, 'gaussian': 2, 'sigmoid': 3, 'laplacian': 4}


@pytest.mark.parametrize('kind', list(KID))
@pytest.mark.parametrize('cfg,n', [('C1', 2000), ('C4', 3000)])
def test_kernel_rows_against_k1(cfg, n, kind):
    """records, does not require, bitwise equality: whether the B200's DMMA rounds as a sequential fma chain"""
    from optiml_b200 import _native as N
    from optiml_b200.runtime import DeviceMatrix, default_context
    spec, X, y = make_config(cfg, n=n)
    ctx = default_context()
    dX = ctx.upload_matrix(X)
    gamma, coef0, degree = 1.0 / (X.shape[1] * X.var()), 0.5, 3.
    ld = N.padded_ld(n)
    rows = np.ascontiguousarray(np.arange(0, n, 7), dtype=np.int64)
    out, K = DeviceMatrix(ctx, len(rows), n, ld), DeviceMatrix(ctx, n, n, ld)
    N.call('svmb200_kernel_rows', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, X.shape[1], KID[kind], gamma, coef0,
           degree, rows.ctypes.data_as(C.c_void_p), len(rows), C.c_void_p(out.dptr), ld)
    N.call('svmb200_gram', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, C.c_void_p(dX.dptr), n, dX.ld, X.shape[1], 1,
           KID[kind], gamma, coef0, degree, None, None, 0.0, 0, n, C.c_void_p(K.dptr), ld)
    got, want = out.to_host(), K.to_host()[rows]
    for m in (out, K, dX):
        m.release()
    np.testing.assert_allclose(got, want, rtol=1e-13, atol=1e-13 * np.abs(want).max())
    print(f'{cfg} {kind}: computed rows bitwise equal to K1: {np.array_equal(got, want)} '
          f'({np.count_nonzero(got != want)} of {got.size} differ)')


@pytest.mark.parametrize('task,kind', [('svc', 'gaussian'), ('svr', 'poly')])
def test_bit_identical_to_the_oracle_and_close_to_libsvm(monkeypatch, task, kind):
    m, X, y = fit(monkeypatch, task, 2000, 'computed')
    o = m.optimizer
    assert o.row_source == 'computed'
    Q = m.obj.device_hessian().to_host()
    r = SO.smo(Q, o.f.q, o.y, o.ub, tol=1e-5, max_iter=10 ** 7)
    assert o.status == r.status == 'optimal' and o.iter == r.iter
    for got, want in ((o.x, r.x), (o.g_x, r.g), (o.f_hist, r.f_hist), (o.gap_hist, r.gap_hist)):
        assert np.array_equal(got, want)
    assert o.rho == r.rho and m.intercept_ == -r.rho
    K, Qh, q, signs, Cb, gamma = SC.problem(task, X, y, kind)
    sk = SC.sklearn_fit(task, X, y, kind, gamma, tol=1e-5)
    SC.check_against_libsvm(task, X, K, Qh, q, signs, Cb, o.x, o.rho, o.gap, 1e-5, sk)
    res, _, _ = fit(monkeypatch, task, 2000, 'resident')
    assert res.optimizer.row_source == 'resident'
    f_c, f_r = o.f_x, res.optimizer.f_x
    assert abs(f_c - f_r) <= 1e-9 * abs(f_r)
    print(f'{task}: computed vs resident fit bitwise equal: {np.array_equal(o.x, res.optimizer.x)}')


def test_cache_size_does_not_change_a_bit(monkeypatch):
    a, _, _ = fit(monkeypatch, 'svc', 2000, 'computed', cache_mb=0)
    b, _, _ = fit(monkeypatch, 'svc', 2000, 'computed')
    oa, ob = a.optimizer, b.optimizer
    assert oa.cache_slots == 0 and oa.cache_hits == 0 and ob.cache_slots == 2000 and ob.cache_misses <= 2000
    for u, v in ((oa.x, ob.x), (oa.g_x, ob.g_x), (oa.f_hist, ob.f_hist), (oa.gap_hist, ob.gap_hist)):
        assert np.array_equal(u, v)
    assert oa.iter == ob.iter and oa.rho == ob.rho


def _pg_fit():
    from optiml_b200.ml.svm import SVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge
    from optiml_b200.opti.constrained import ProjectedGradient
    spec, X, y = make_config('C1', n=1500)
    m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, reg_intercept=True, optimizer=ProjectedGradient,
            max_iter=300, tol=1e-6).fit(X, y)
    return m.alphas_.copy(), float(m.intercept_)


def test_large_fit_beyond_hbm_and_others_unchanged(monkeypatch):
    monkeypatch.delenv('SVMB200_SMO_ROWS', raising=False)
    monkeypatch.delenv('SVMB200_SMO_CACHE_MB', raising=False)
    pg0 = _pg_fit()
    res0, _, _ = fit(monkeypatch, 'svc', 1500, 'resident')
    monkeypatch.delenv('SVMB200_SMO_ROWS', raising=False)
    n, tol = 200_000, 1e-3
    from optiml_b200.ml.svm import SVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge
    spec, X, y = make_config('C5', n=n)
    m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=10 ** 7).fit(X, y)
    o = m.optimizer
    assert o.row_source == 'computed' and o.status == 'optimal' and o.gap < tol
    a, ys = o.x, o.y
    assert np.all(a >= 0) and np.all(a <= o.ub)
    assert abs(ys @ a) <= 1e-10 * n
    G = m.obj.device_hessian().product(a) + o.f.q   # K6, independent of the solver's rows
    np.testing.assert_allclose(G, o.g_x, rtol=0, atol=1e-8 * max(1.0, np.abs(o.g_x).max()))
    up = np.where(ys > 0, a < o.ub, a > 0)
    low = np.where(ys > 0, a > 0, a < o.ub)
    gap = np.max(-(ys * G)[up]) - np.min(-(ys * G)[low])
    assert gap <= tol
    print(f'n = {n}: {o.iter} iterations, {o.device_ms / 1e3:.2f} s solve, cache {o.cache_slots} slots, '
          f'hit rate {o.cache_hits / max(o.cache_hits + o.cache_misses, 1):.4f}, KKT gap from K6 {gap:.3e}')
    m.obj.release()
    res1, _, _ = fit(monkeypatch, 'svc', 1500, 'resident')
    for u, v in ((res0.optimizer.x, res1.optimizer.x), (res0.optimizer.gap_hist, res1.optimizer.gap_hist)):
        assert np.array_equal(u, v)
    pg1 = _pg_fit()
    assert np.array_equal(pg0[0], pg1[0]) and pg0[1] == pg1[1]
