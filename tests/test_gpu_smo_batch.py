"""SMO on signed views of one unsigned M and the SMO batch (csrc/k_smo.cuh K14, svmb200_smo_run_batch,
ml/multiclass.py) on the B200: bit for bit against single solves and against sklearn's clone-per-class fits, at sizes
with several CTAs per problem; the reference's iris recipe; C4's inputs in four classes against the KKT conditions."""
import numpy as np
import pytest

import smo_batch_checks as SB
from optiml_b200.configs import make_config

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('kind', ['gaussian', 'linear', 'poly'])
def test_signed_view_equals_k1_signed_q(kind):
    from optiml_b200.ml.svm.kernels import GaussianKernel, LinearKernel, PolyKernel
    kernel = {'gaussian': GaussianKernel(), 'linear': LinearKernel(), 'poly': PolyKernel(degree=3)}[kind]
    spec, X, y = make_config('C1', n=3000)
    a, b, _ = SB.signed_view_against_k1(SB.svc(kernel), X, np.where(y > 0, 1.0, -1.0), tol=1e-3)
    assert a.status == 'optimal'
    SB.assert_same_solve(a, b)


def _shared_m(n, svr=False):
    spec, X, y = make_config('C2' if svr else 'C1', n=n)
    est = SB.svr() if svr else SB.svc()
    H = est._build_hessian(X, None, 'svr' if svr else 'plain', None, 0.0)
    est._train_X_device[0].release()
    return X, y, H


# n = 6 000: single-fit grid 47 CTAs, g_min = 2
@pytest.mark.parametrize('count,sms,chunk', [
    (4, None, None),   # 37 CTAs each
    (6, 10, 300),      # a cap below count x g_min: five at a time, the sixth waits; short chunks regrid
    (3, 2, 500),       # one problem at a time
])
def test_batch_equals_each_solvers_own_run(monkeypatch, count, sms, chunk):
    from optiml_b200.runtime import default_context
    if sms:
        monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', str(sms))
    if chunk:
        monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', str(chunk))
    X, y, H = _shared_m(6000)
    try:
        SB.check_batch_equals_single_runs(lambda: SB.batch_problems(default_context(), H, X, count, tol=1e-3))
    finally:
        H.release()


def test_forced_waves_of_large_problems(monkeypatch):
    """C4-sized problems need 11 CTAs each (slices of at most 4 714 variables): a cap of 30 SMs holds two at a time"""
    from optiml_b200.runtime import default_context
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '30')
    X, y, H = _shared_m(50000)
    try:
        SB.check_batch_equals_single_runs(
            lambda: SB.batch_problems(default_context(), H, X, 3, tol=1e-2, max_iters={0: 3000, 1: 2000, 2: 4000}))
    finally:
        H.release()


def test_svr_multi_target():
    from sklearn.multioutput import MultiOutputRegressor as SklearnMOR
    from optiml_b200.ml.multiclass import MultiOutputRegressor
    spec, X, y = make_config('C2', n=4000)
    Y = np.stack([y, np.roll(y, 11), 0.5 * y + 1.0], axis=1)
    ours = MultiOutputRegressor(SB.svr(tol=1e-3)).fit(X, Y)
    theirs = SklearnMOR(SB.svr(tol=1e-3)).fit(X, Y)
    SB.compare_estimators(ours.estimators_, theirs.estimators_, X)
    assert np.array_equal(ours.predict(X), theirs.predict(X))
    SB.assert_one_shared_matrix(ours.estimators_)


def test_iris_one_vs_rest(golden):
    """the reference's recipe (ml/tests/test_svc.py:96-115) with optimizer='smo', on one M"""
    from optiml_b200.ml.multiclass import OneVsRestClassifier
    from optiml_b200.ml.svm.kernels import gaussian
    g = golden('iris_ovr')
    ovr = OneVsRestClassifier(SB.svc(gaussian)).fit(g['X_train'], g['y_train'])
    assert ovr.score(g['X_test'], g['y_test']) >= 0.97
    assert all(e.optimizer.status == 'optimal' for e in ovr.estimators_)
    SB.assert_one_shared_matrix(ovr.estimators_)
    SB.compare_ovr(SB.svc(gaussian), g['X_train'], g['y_train'])


def test_c4_four_classes_equal_clone_per_class_and_reach_the_kkt_conditions():
    tol = 1e-3
    spec, X, y2 = make_config('C4')
    y = SB.quantile_classes(X, 4)
    ours, _ = SB.compare_ovr(SB.svc(tol=tol, max_iter=10 ** 7), X, y)
    SB.assert_one_shared_matrix(ours.estimators_)
    for c, m in zip(ours.classes_, ours.estimators_):
        o = m.optimizer
        a, G, s = o.x, o.g_x, o.y
        assert np.array_equal(s, np.where(y == c, 1.0, -1.0))
        assert o.status == 'optimal' and o.gap < tol
        assert np.all(a >= 0) and np.all(a <= 1.0)
        assert abs(s @ a) <= 1e-10 * 1.0 * len(y)
        Qa = m.obj.device_hessian().product(a)   # one masked product on the signed view
        f = 0.5 * a @ Qa - a.sum()
        assert abs(o.f_x - f) <= 1e-10 * abs(f)
        minus_yG = -s * G
        up = np.where(s > 0, a < 1.0, a > 0)
        low = np.where(s > 0, a > 0, a < 1.0)
        assert minus_yG[up].max() - minus_yG[low].min() <= tol
