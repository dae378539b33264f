"""SMO on signed views of one unsigned M and the SMO batch (csrc/k_smo.cuh K14, svmb200_smo_run_batch,
ml/multiclass.py) on the host emulation of the CUDA runtime (tests/cuda_emu), which reports 148 SMs: small SM caps and
short chunks exercise waves and regridding at small n."""
import ctypes as C
import warnings

import numpy as np
import pytest
from sklearn.datasets import load_iris, make_classification
from sklearn.exceptions import ConvergenceWarning

import smo_batch_checks as SB
from emu import emulated_device
from optiml_b200 import _native as N
from optiml_b200.configs import make_config


def zero_rich_inputs(n=120, d=12, seed=3):
    """sparse 0/1 rows: many pairs are orthogonal, so linear and polynomial Grams hold exact zeros (and a Gaussian
    Gram with gamma = 200 underflows to zero from a squared distance of 4 on)"""
    rng = np.random.default_rng(seed)
    return (rng.random((n, d)) < 0.15).astype(np.float64)


@pytest.mark.parametrize('kind', ['gaussian', 'linear', 'poly'])
def test_signed_view_equals_k1_signed_q(kind):
    from optiml_b200.ml.svm.kernels import GaussianKernel, LinearKernel, PolyKernel
    kernel = {'gaussian': GaussianKernel(gamma=200.0), 'linear': LinearKernel(), 'poly': PolyKernel(degree=3)}[kind]
    X = zero_rich_inputs()
    ys = np.where(X[:, 0] + X[:, 1] + np.arange(len(X)) % 3 > 1, 1.0, -1.0)
    with emulated_device() as lib:
        a, b, Q = SB.signed_view_against_k1(SB.svc(kernel), X, ys)
        assert lib.emu_sticky_error() == 0
    zeros = Q == 0
    assert zeros.any() and np.signbit(Q[zeros]).any() and (~np.signbit(Q[zeros])).any()   # both signed zeros
    assert a.status == 'optimal' and a.row_source == b.row_source == 'resident'
    SB.assert_same_solve(a, b)
    assert a.rho == b.rho


def test_svr_signed_view_equals_the_svr_read():
    spec, X, y = make_config('C2', n=70)
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        est = SB.svr()
        H = est._build_hessian(X, None, 'svr', None, 0.0)
        est._train_X_device[0].release()
        n = len(y)
        e, q = np.hstack((np.ones(n), -np.ones(n))), np.hstack((-y, y)) + 0.1
        got = []
        for signed in (False, True):
            p = SB.Problem(ctx, H, e, q, 1e-5, 10 ** 6, svr=True, signed=signed)
            got.append(p.run() + p.result())
            p.destroy()
        H.release()
        assert lib.emu_sticky_error() == 0
    assert got[0][:2] == got[1][:2] and N.STATUS[got[0][1]] == 'optimal'
    for u, v in zip(got[0][2:], got[1][2:]):
        assert np.array_equal(u, v)


def _shared_m(n=300, svr=False):
    """K1's unsigned M (bias 0) of C1 / C2 inputs on the emulated device"""
    spec, X, y = make_config('C2' if svr else 'C1', n=n)
    est = SB.svr() if svr else SB.svc()
    H = est._build_hessian(X, None, 'svr' if svr else 'plain', None, 0.0)
    est._train_X_device[0].release()
    return X, y, H


@pytest.mark.parametrize('count,sms,chunk', [
    (1, None, None),
    (3, None, None),      # every problem on its single-fit grid of 3 CTAs
    (4, 2, None),         # one CTA each, two at a time: the others wait for a later wave
    (5, 7, 13),           # uneven split, short chunks: early finishers give their SMs to the others
    (6, 4, 40),
])
def test_batch_equals_each_solvers_own_run(monkeypatch, count, sms, chunk):
    if sms:
        monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', str(sms))
    if chunk:
        monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', str(chunk))
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        X, y, H = _shared_m()
        want = SB.check_batch_equals_single_runs(lambda: SB.batch_problems(ctx, H, X, count), lib)
        H.release()
        assert lib.emu_sticky_error() == 0
    if count > 1:
        assert len({w[0] for w in want}) > 1   # the problems need different numbers of iterations


@pytest.mark.parametrize('order', [0, 1, 2])
def test_batch_with_one_problem_stopped_at_max_iter_under_every_schedule(monkeypatch, order):
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '5')
    monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', '16')
    with emulated_device(order=order, seed=11) as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        X, y, H = _shared_m()
        want = SB.check_batch_equals_single_runs(lambda: SB.batch_problems(ctx, H, X, 3, max_iters={1: 37}), lib)
        H.release()
        assert lib.emu_sticky_error() == 0
    assert want[1][0] == 37 and N.STATUS[want[1][1]] == 'stopped'
    assert N.STATUS[want[0][1]] == N.STATUS[want[2][1]] == 'optimal' and want[0][0] > 37 and want[2][0] > 37


def test_svr_batch_on_a_shared_m(monkeypatch):
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '3')
    monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', '50')
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        X, y, H = _shared_m(n=80, svr=True)
        Y = np.stack([y, np.roll(y, 7), 0.5 * y + 1.0], axis=1)
        SB.check_batch_equals_single_runs(lambda: SB.batch_problems(ctx, H, X, 3, svr_targets=Y), lib)
        H.release()
        assert lib.emu_sticky_error() == 0


def test_abi_refusals():
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        X, y, H = _shared_m(n=60)
        X2, y2, H2 = _shared_m(n=60)
        n = H.n
        a, b, c = SB.batch_problems(ctx, H, X, 3)
        other = SB.batch_problems(ctx, H2, X2, 1)[0]
        svr_view = SB.Problem(ctx, H, np.hstack((np.ones(n), -np.ones(n))), -np.ones(2 * n), 1e-5, 100, svr=True,
                              signed=True)
        pg = C.c_void_p()
        N.call('svmb200_pg_create', ctx.handle, C.c_void_p(H.matrix.dptr), n, H.ld, 0, n, N.HESSIAN_PLAIN,
               N.ptr(-np.ones(n)), None, N.ptr(np.ones(n)), None, 1e-6, 10, C.byref(pg))
        dX = ctx.upload_matrix(X)
        rows = C.c_void_p()
        N.call('svmb200_smo_create_rows', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, X.shape[1], 2, 0.1, 0.0, 3.0,
               N.HESSIAN_PLAIN, N.ptr(np.where(y > 0, 1.0, -1.0)), N.ptr(-np.ones(n)), N.ptr(np.ones(n)), 1e-3, 100, 0,
               C.byref(rows))

        def refused(handles, text):
            arr = (C.c_void_p * len(handles))(*[h.value for h in handles])
            assert lib.svmb200_smo_run_batch(arr, len(handles), None, None) == 1   # SVMB200_ERR_ARG
            assert text in lib.svmb200_last_error()

        refused([a.h, other.h], b'share the resident matrix')
        refused([a.h, svr_view.h], b'share the resident matrix')
        refused([a.h, rows], b'computed rows')
        refused([a.h, pg], b'SMO solvers only')
        refused([a.h, b.h, a.h], b'listed twice')
        refused([C.c_void_p()], b'null solver')
        arr = (C.c_void_p * 2)(a.h.value, b.h.value)
        assert lib.svmb200_pg_run_batch(arr, 2, None, None) == 1
        assert b'SMO solvers have no lockstep batch' in lib.svmb200_last_error()
        c.run()
        refused([a.h, c.h], b'have not run yet')
        assert SB.run_batch([a, b])[0] == 0
        refused([a.h], b'have not run yet')
        for p in (a, b, c, other, svr_view):
            p.destroy()
        for h in (pg, rows):
            lib.svmb200_pg_destroy(h)
        for m in (dX, H, H2):
            m.release()
        assert lib.emu_sticky_error() == 0


def test_batch_returns_its_allocations(monkeypatch):
    from optiml_b200.runtime import Context
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '2')
    monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', '700')   # the histories grow past their first 1 024 states
    with emulated_device() as lib:
        base = lib.emu_live_allocations()
        ctx = Context(device=0)
        from optiml_b200.runtime import DeviceHessian
        spec, X, y = make_config('C1', n=90)
        K = np.exp(-((X[:, None] - X[None]) ** 2).sum(-1) / X.shape[1])
        H = DeviceHessian.from_host(ctx, K)
        live = None
        for _ in range(2):   # the first batch also takes the context's scratch and grid barrier, which stay with it
            probs = []
            for b in range(3):
                ys = np.where(np.roll(y, 5 * b) > 0, 1.0, -1.0)
                probs.append(SB.Problem(ctx, H, ys, -np.ones(90), 0.0, 1500 + b))   # tol 0: every problem runs to max_iter
            rc, iters, _ = SB.run_batch(probs, lib)
            assert rc == 0 and iters == [1500, 1501, 1502]
            for p in probs:
                p.destroy()
            assert live is None or lib.emu_live_allocations() == live
            live = lib.emu_live_allocations()
        H.release()
        ctx.trim()
        ctx._finalizer()
        assert lib.emu_live_allocations() == base
        assert lib.emu_sticky_error() == 0


# ------------------------------------------------------------------ estimators
def _four_classes(n=160):
    X, y = make_classification(n_samples=n, n_features=6, n_informative=4, n_redundant=0, n_classes=4,
                               n_clusters_per_class=1, random_state=2)
    return X, y


@pytest.mark.parametrize('data', ['iris', 'four_classes'])
def test_one_vs_rest_equals_clone_per_class(data):
    X, y = load_iris(return_X_y=True) if data == 'iris' else _four_classes()
    with emulated_device() as lib:
        ours, theirs = SB.compare_ovr(SB.svc(tol=1e-3), X, y)
        SB.assert_one_shared_matrix(ours.estimators_)
        assert all('batch' not in e.fit_times_ for e in theirs.estimators_)
        assert lib.emu_sticky_error() == 0


def test_one_vs_rest_with_a_class_stopped_at_max_iter():
    X, y = _four_classes()
    with emulated_device() as lib:
        from optiml_b200.ml.multiclass import OneVsRestClassifier
        free = OneVsRestClassifier(SB.svc(tol=1e-3)).fit(X, y)
        iters = sorted(e.optimizer.iter for e in free.estimators_)
        assert iters[0] < iters[-1]
        ours, _ = SB.compare_ovr(SB.svc(tol=1e-3, max_iter=iters[-1] - 1), X, y)
        status = [e.optimizer.status for e in ours.estimators_]
        assert 'stopped' in status and 'optimal' in status
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter('always')
            OneVsRestClassifier(SB.svc(tol=1e-3, max_iter=iters[-1] - 1)).fit(X, y)
        assert sum(issubclass(x.category, ConvergenceWarning) for x in w) == status.count('stopped')
        assert lib.emu_sticky_error() == 0


def test_multi_output_svr_equals_one_fit_per_target():
    from sklearn.multioutput import MultiOutputRegressor as SklearnMOR
    from optiml_b200.ml.multiclass import MultiOutputRegressor
    spec, X, y = make_config('C2', n=90)
    Y = np.stack([y, np.roll(y, 11), 0.5 * y + 1.0], axis=1)
    with emulated_device() as lib:
        ours = MultiOutputRegressor(SB.svr(tol=1e-4)).fit(X, Y)
        theirs = SklearnMOR(SB.svr(tol=1e-4)).fit(X, Y)
        SB.compare_estimators(ours.estimators_, theirs.estimators_, X)
        assert np.array_equal(ours.predict(X), theirs.predict(X))
        SB.assert_one_shared_matrix(ours.estimators_)
        assert lib.emu_sticky_error() == 0


def test_computed_rows_fall_back_to_clone_per_class(monkeypatch):
    monkeypatch.setenv('SVMB200_SMO_ROWS', 'computed')
    X, y = load_iris(return_X_y=True)
    with emulated_device() as lib:
        ours, theirs = SB.compare_ovr(SB.svc(tol=1e-3), X, y)
        assert all(e.optimizer.row_source == 'computed' and 'batch' not in e.fit_times_ for e in ours.estimators_)
        assert lib.emu_sticky_error() == 0


def test_verbose_falls_back_to_clone_per_class(capsys):
    X, y = load_iris(return_X_y=True)
    with emulated_device() as lib:
        ours, theirs = SB.compare_ovr(SB.svc(tol=1e-3, verbose=True), X, y)
        assert all('batch' not in e.fit_times_ for e in ours.estimators_)
        assert lib.emu_sticky_error() == 0


def test_sharded_context_is_refused_before_any_device_work(monkeypatch):
    from optiml_b200 import runtime
    from optiml_b200.ml.multiclass import MultiOutputRegressor, OneVsRestClassifier

    class ShardedContext:   # what default_context() is under torchrun with two ranks; any device call would fail
        nranks, group = 2, None
    monkeypatch.setattr(runtime, '_default_ctx', ShardedContext())
    X, y = load_iris(return_X_y=True)
    with pytest.raises(NotImplementedError, match='one GPU'):
        OneVsRestClassifier(SB.svc()).fit(X, y)
    with pytest.raises(NotImplementedError, match='one GPU'):
        MultiOutputRegressor(SB.svr()).fit(X, np.stack([X[:, 0], X[:, 1]], axis=1))
