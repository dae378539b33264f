"""Shrinking in K11 / K12 / K14 (csrc/k_smo.cuh, the SHRINK instantiations) on the host emulation of the CUDA runtime
(tests/cuda_emu): estimator fits with ``shrinking=True`` are bit-identical to tests/smo_shrinking_oracle.py replayed on
the matrix the kernel read -- resident, signed-view and computed rows, every grid, schedule, cache and call pattern --
and the shared one-vs-rest / grid-search paths equal sklearn's clone path.  The oracle itself is checked against the KKT
conditions and sklearn's SVC / SVR."""
import ctypes as C
import gc
import warnings

import numpy as np
import pytest
from sklearn.base import clone
from sklearn.exceptions import ConvergenceWarning

import smo_batch_checks as SB
import smo_cv_checks as CV
import smo_shrinking_oracle as SSO
from emu import emulated_device
from oracle import smo_oracle as SO
from optiml_b200.configs import make_config


def estimator(task, max_iter=10 ** 6, tol=1e-5, **kw):
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    if task == 'svc':
        return SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=max_iter,
                   **kw)
    return SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo',
               tol=tol, max_iter=max_iter, **kw)


def data(task, n):
    return make_config('C1' if task == 'svc' else 'C2', n=n)[1:]


def fit(monkeypatch, task, n, grid, rows='resident', cache_mb=None, order=0, max_iter=10 ** 6, shrinking=True):
    monkeypatch.setenv('SVMB200_SMO_GRID', str(grid))
    monkeypatch.setenv('SVMB200_SMO_ROWS', rows)
    if cache_mb is None:
        monkeypatch.delenv('SVMB200_SMO_CACHE_MB', raising=False)
    else:
        monkeypatch.setenv('SVMB200_SMO_CACHE_MB', repr(cache_mb))
    X, y = data(task, n)
    m = estimator(task, max_iter=max_iter, shrinking=shrinking)
    with emulated_device(order=order, seed=5) as lib:
        m.fit(X, y)
        Q = m.obj.device_hessian().to_host()
        assert lib.emu_sticky_error() == 0
    assert m.optimizer.row_source == rows
    return m, Q


def outcome(o):
    return o.x, o.g_x, o.f_hist, o.gap_hist, o.iter, o.status, o.rho


def assert_same(a, b):
    for u, v in zip(outcome(a), outcome(b)):
        assert np.array_equal(u, v)


def assert_oracle(o, Q, tol=1e-5, max_iter=10 ** 6):
    r = SSO.smo(Q, o.f.q, o.y, o.ub, tol=tol, max_iter=max_iter, shrinking=True)
    assert o.status == r.status and o.iter == r.iter
    for got, want in ((o.x, r.x), (o.g_x, r.g), (o.f_hist, r.f_hist), (o.gap_hist, r.gap_hist)):
        assert np.array_equal(got, want)
    assert o.rho == r.rho and o.f_x == r.f_x
    assert (o.active_, o.shrink_checks, o.reconstructions) == (r.active, r.checks, r.reconstructions)
    return r


# ------------------------------------------------------------------ the oracle
def _kkt_gap(r, Q, q, y, C):
    G = Q @ r.x + q   # the full G, recomputed
    up = np.where(y > 0, r.x < C, r.x > 0)
    low = np.where(y > 0, r.x > 0, r.x < C)
    return np.max(-y[up] * G[up]) - np.min(-y[low] * G[low]), G


@pytest.mark.parametrize('task,n', [('svc', 300), ('svr', 150)])
def test_oracle_meets_kkt_and_matches_sklearn(task, n):
    from sklearn.svm import SVC, SVR
    from oracle import svm_oracle as O
    X, y = data(task, n)
    gamma = 1.0 / (X.shape[1] * X.var())
    if task == 'svc':
        ys = np.where(y > 0, 1.0, -1.0)
        K = O.gaussian_kernel(X, gamma=gamma)
        Q, q, sgn = ys[:, None] * K * ys[None, :], -np.ones(n), ys
        ref = SVC(C=1.0, kernel='rbf', gamma=gamma, tol=1e-5, shrinking=True).fit(X, y)
        coef = np.zeros(n)
        coef[ref.support_] = ref.dual_coef_.ravel()
        ref_obj = 0.5 * coef @ K @ coef - np.abs(coef).sum()
    else:
        K = O.kernel_matrix('poly', X, degree=3, gamma=gamma, coef0=0.0)
        Q = np.block([[K, -K], [-K, K]])
        q, sgn = np.concatenate([0.1 - y, 0.1 + y]), np.repeat([1.0, -1.0], n)
        ref = SVR(C=1.0, kernel='poly', degree=3, gamma=gamma, coef0=0.0, epsilon=0.1, tol=1e-5).fit(X, y)
        coef = np.zeros(n)
        coef[ref.support_] = ref.dual_coef_.ravel()
        ref_obj = 0.5 * coef @ K @ coef + 0.1 * np.abs(coef).sum() - coef @ y
    r = SSO.smo(Q, q, sgn, 1.0, tol=1e-5, shrinking=True)
    plain = SO.smo(Q, q, sgn, 1.0, tol=1e-5)
    assert r.status == 'optimal' and r.checks >= 1
    gap, G = _kkt_gap(r, Q, q, sgn, np.ones_like(q))
    assert gap < 1e-5
    np.testing.assert_allclose(r.g, G, rtol=0, atol=1e-10)   # the G it returns is the full, reconstructed G
    np.testing.assert_allclose(r.f_x, ref_obj, rtol=1e-6)
    np.testing.assert_allclose(r.f_x, plain.f_x, rtol=1e-6)


@pytest.mark.parametrize('task,n', [('svc', 2000), ('svr', 400)])
def test_oracle_shrinks_on_c1_and_svr_problems(task, n):
    """shrinking engages (variables set aside, G rebuilt) and ends at the plain solver's optimum.  The trajectories
    may still agree: a variable set aside is one WSS2 would not have selected until the gap closes."""
    from oracle import svm_oracle as O
    X, y = data(task, n)
    if task == 'svc':
        ys = np.where(y > 0, 1.0, -1.0)
        Q, q, sgn = ys[:, None] * O.gaussian_kernel(X) * ys[None, :], -np.ones(n), ys
    else:
        K = O.kernel_matrix('poly', X, degree=3, gamma=1.0 / X.shape[1], coef0=0.0)
        Q, q, sgn = np.block([[K, -K], [-K, K]]), np.concatenate([0.1 - y, 0.1 + y]), np.repeat([1.0, -1.0], n)
    tol = 1e-3 if task == 'svc' else 1e-5   # enough states for a check (P = min(l, 1000))
    r = SSO.smo(Q, q, sgn, 1.0, tol=tol, shrinking=True)
    plain = SO.smo(Q, q, sgn, 1.0, tol=tol)
    assert r.status == plain.status == 'optimal'
    assert r.checks >= 1 and r.active < len(q) // 2 and r.reconstructions >= 1
    gap, G = _kkt_gap(r, Q, q, sgn, np.ones_like(q))
    assert gap < tol
    np.testing.assert_allclose(r.g, G, rtol=0, atol=1e-9)
    np.testing.assert_allclose(r.f_x, plain.f_x, rtol=1e-4)


def test_oracle_without_shrinking_is_the_plain_oracle():
    X, y = data('svc', 60)
    ys = np.where(y > 0, 1.0, -1.0)
    from oracle import svm_oracle as O
    Q = ys[:, None] * O.gaussian_kernel(X) * ys[None, :]
    a, b = SSO.smo(Q, -1.0, ys, 1.0, tol=1e-5), SO.smo(Q, -1.0, ys, 1.0, tol=1e-5)
    assert np.array_equal(a.x, b.x) and np.array_equal(a.gap_hist, b.gap_hist)


# ------------------------------------------------------------------ K11 / K12 with shrinking
@pytest.mark.parametrize('task,n', [('svc', 131), ('svc', 257), ('svr', 97)])
@pytest.mark.parametrize('grid', [1, 3, 8])
@pytest.mark.parametrize('rows', ['resident', 'computed'])
def test_estimator_fit_is_bit_identical_to_the_oracle(monkeypatch, task, n, grid, rows):
    m, Q = fit(monkeypatch, task, n, grid, rows)
    r = assert_oracle(m.optimizer, Q)
    assert r.status == 'optimal' and r.checks >= 1
    assert m.intercept_ == -r.rho


@pytest.mark.parametrize('cache_mb', [0, 0.003, 1])   # no cache, a small set-associative one, every row
def test_computed_rows_with_every_cache_follow_the_oracle(monkeypatch, cache_mb):
    m, Q = fit(monkeypatch, 'svc', 257, 3, 'computed', cache_mb=cache_mb)
    assert_oracle(m.optimizer, Q)
    o = m.optimizer
    assert (o.cache_slots == 0) == (cache_mb == 0)


@pytest.mark.parametrize('order', [1, 2])
@pytest.mark.parametrize('rows', ['resident', 'computed'])
def test_thread_and_block_schedules_do_not_change_a_bit(monkeypatch, order, rows):
    a, _ = fit(monkeypatch, 'svc', 257, 8, rows)
    b, _ = fit(monkeypatch, 'svc', 257, 8, rows, order=order)
    assert_same(a.optimizer, b.optimizer)


@pytest.mark.parametrize('rows', ['resident', 'computed'])
def test_one_iteration_calls_equal_one_run(monkeypatch, rows):
    """a generic callback makes the solver synchronise at every state (one launch per state): the counter, the flags
    and the unshrink state carry across launches"""
    from optiml_b200.ml.svm.smo import SMO
    monkeypatch.setenv('SVMB200_SMO_GRID', '3')
    monkeypatch.setenv('SVMB200_SMO_ROWS', rows)
    X, y = data('svc', 131)
    m = estimator('svc', shrinking=True, tol=1e-6)
    seen = []
    with emulated_device() as lib:
        m.fit(X, y)
        o = SMO(quad=m.obj, y=m.optimizer.y, C=1., tol=1e-6, max_iter=10 ** 6, shrinking=True,
                callback=lambda opt: seen.append(opt.iter)).minimize()
        assert lib.emu_sticky_error() == 0
    assert m.optimizer.shrink_checks >= 1
    assert seen == list(range(o.iter + 1))
    assert_same(o, m.optimizer)
    assert (o.active_, o.shrink_checks, o.reconstructions) == \
        (m.optimizer.active_, m.optimizer.shrink_checks, m.optimizer.reconstructions)


@pytest.mark.parametrize('rows', ['resident', 'computed'])
def test_max_iter_stop_returns_the_reconstructed_g(monkeypatch, rows):
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        m, Q = fit(monkeypatch, 'svc', 257, 3, rows, max_iter=400)
    assert any(issubclass(x.category, ConvergenceWarning) for x in w)
    o = m.optimizer
    r = assert_oracle(o, Q, max_iter=400)
    assert o.status == 'stopped' and o.iter == 400 and r.checks >= 1
    np.testing.assert_allclose(o.g_x, Q @ o.x + o.f.q, rtol=0, atol=1e-10)


def test_shrinking_off_keeps_the_plain_bits(monkeypatch):
    a, Q = fit(monkeypatch, 'svr', 97, 3, shrinking=False)
    r = SO.smo(Q, a.optimizer.f.q, a.optimizer.y, a.optimizer.ub, tol=1e-5, max_iter=10 ** 6)
    assert np.array_equal(a.optimizer.x, r.x) and np.array_equal(a.optimizer.gap_hist, r.gap_hist)
    assert a.optimizer.shrink_checks == 0 and a.optimizer.active_ == 2 * 97


# ------------------------------------------------------------------ K14, folds, estimators
def test_a_batch_mixing_shrinking_and_plain_problems_equals_their_own_runs(monkeypatch):
    from optiml_b200 import _native as N
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '5')
    monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', '64')
    X, y = data('svc', 300)
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        est = SB.svc()
        H = est._build_hessian(X, None, 'plain', None, 0.0)
        est._train_X_device[0].release()
        n = H.n
        ys = np.where(y > 0, 1.0, -1.0)

        def problems():
            out = []
            for b, (shrink, c) in enumerate([(True, 1.0), (False, 1.0), (True, 3.0), (True, 0.5)]):
                p = SB.Problem(ctx, H, ys, -c * np.ones(n), 1e-5, 300 if b == 3 else 10 ** 6)
                if shrink:
                    N.call('svmb200_smo_set_shrinking', p.h, 1)
                out.append(p)
            return out

        SB.check_batch_equals_single_runs(problems, lib)
        H.release()
        assert lib.emu_sticky_error() == 0


@pytest.mark.parametrize('sms,chunk', [(None, None), (3, 16)])
def test_folds_with_shrinking_equal_their_own_fits(monkeypatch, sms, chunk):
    if sms:
        monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', str(sms))
        monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', str(chunk))
    X, y = data('svc', 260)
    rows = CV.ragged_rows(len(y), 3)
    with emulated_device() as lib:
        CV.check_folds_equal_own_fits(SB.svc(tol=1e-5, shrinking=True), X, y, rows,
                                      params=[{}, {'C': 4.0}, {'shrinking': False}])
        assert lib.emu_sticky_error() == 0


def test_svr_folds_with_shrinking_equal_their_own_fits(monkeypatch):
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '4')
    monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', '40')
    X, y = data('svr', 120)
    with emulated_device() as lib:
        CV.check_folds_equal_own_fits(SB.svr(tol=1e-5, shrinking=True), X, y, CV.ragged_rows(len(y), 2, seed=1))
        assert lib.emu_sticky_error() == 0


@pytest.mark.parametrize('sms,chunk', [(None, None), (4, 32)])
def test_one_vs_rest_with_shrinking_equals_clone_per_class(monkeypatch, sms, chunk):
    from sklearn.datasets import make_classification
    if sms:
        monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', str(sms))
        monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', str(chunk))
    X, y = make_classification(n_samples=240, n_features=6, n_informative=4, n_redundant=0, n_classes=3,
                               n_clusters_per_class=1, random_state=2)
    with emulated_device() as lib:
        ours, theirs = SB.compare_ovr(SB.svc(tol=1e-5, shrinking=True), X, y)
        SB.assert_one_shared_matrix(ours.estimators_)
        assert any(e.optimizer.shrink_checks > 0 for e in ours.estimators_)
        assert lib.emu_sticky_error() == 0


@pytest.mark.parametrize('sms,chunk', [(None, None), (3, 24)])
def test_grid_search_over_shrinking_equals_sklearns(monkeypatch, sms, chunk):
    if sms:
        monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', str(sms))
        monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', str(chunk))
    X, y = data('svc', 240)
    with emulated_device() as lib:
        ours, theirs = CV.grid_search_both(SB.svc(tol=1e-5), {'C': [0.5, 2.0], 'shrinking': [False, True]}, X, y,
                                           cv=3)
        assert ours.best_estimator_.shrinking == theirs.best_estimator_.shrinking
        assert lib.emu_sticky_error() == 0


# ------------------------------------------------------------------ the interface
def test_estimator_keyword_clone_params_and_pickle():
    import pickle
    m = estimator('svc', shrinking=True)
    assert m.get_params()['shrinking'] is True and clone(m).shrinking is True
    assert pickle.loads(pickle.dumps(m)).shrinking is True
    assert estimator('svr').get_params()['shrinking'] is False
    from optiml_b200.ml.svm import DualSVC, DualSVR
    assert DualSVC(shrinking=True).shrinking and DualSVR().get_params()['shrinking'] is False


def test_shrinking_without_smo_is_refused_at_fit():
    from optiml_b200.ml.svm import DualSVC
    X, y = data('svc', 40)
    m = DualSVC(shrinking=True, max_iter=5)
    with pytest.raises(ValueError, match="optimizer='smo'"):
        m.fit(X, y)


def test_set_shrinking_after_a_run_is_refused_and_allocations_are_released(monkeypatch):
    from optiml_b200 import _native as N
    monkeypatch.setenv('SVMB200_SMO_ROWS', 'computed')
    X, y = data('svc', 90)
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        base = lib.emu_live_allocations()
        ctx = default_context()
        ys = np.where(y > 0, 1.0, -1.0)
        dX = ctx.upload_matrix(X)
        h = C.c_void_p()
        N.call('svmb200_smo_create_rows', ctx.handle, C.c_void_p(dX.dptr), len(y), dX.ld, X.shape[1], 2, 0.2, 0.0, 3.0,
               N.HESSIAN_PLAIN, N.ptr(ys), N.ptr(-np.ones(len(y))), N.ptr(np.ones(len(y))), 1e-5, 10 ** 6, 1 << 16,
               C.byref(h))
        N.call('svmb200_smo_set_shrinking', h, 1)
        N.call('svmb200_smo_set_shrinking', h, 0)
        N.call('svmb200_smo_set_shrinking', h, 1)
        it, st = C.c_int64(0), C.c_int(0)
        N.call('svmb200_pg_run', h, 0, C.byref(it), C.byref(st))   # state 0 only: a run has started
        assert lib.svmb200_smo_set_shrinking(h, 0) != 0
        assert b'already run' in lib.svmb200_last_error()
        N.call('svmb200_pg_run', h, -1, C.byref(it), C.byref(st))
        active, checks, recons = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        N.call('svmb200_smo_shrink_stats', h, C.byref(active), C.byref(checks), C.byref(recons))
        assert checks.value >= 0 and 0 < active.value <= len(y)
        lib.svmb200_pg_destroy(h)
        dX.release()
        gc.collect()
        ctx.trim()
        ctx._finalizer()
        assert lib.emu_live_allocations() == base
        assert lib.emu_sticky_error() == 0
