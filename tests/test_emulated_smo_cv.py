"""Cross-validation folds as masked problems on one shared M (svmb200_smo_create_subset, fit_shared_gram with training
rows, optiml_b200/model_selection.py) on the host emulation of the CUDA runtime (tests/cuda_emu)."""
import ctypes as C
import gc

import numpy as np
import pytest
from sklearn.datasets import load_iris
from sklearn.model_selection import KFold, StratifiedKFold

import smo_batch_checks as SB
import smo_cv_checks as CV
from emu import emulated_device
from optiml_b200 import _native as N
from optiml_b200.configs import make_config


def _binary(n=90, seed=0):
    spec, X, y = make_config('C1', n=n)
    return X, np.where(SB.quantile_classes(X, 2, seed) > 0, 1, -1)


@pytest.mark.parametrize('kind', ['linear', 'poly', 'gaussian', 'laplacian', 'sigmoid'])
@pytest.mark.parametrize('layout', ['plain', 'svr'])
def test_sub_gram_is_the_gram_of_the_rows(kind, layout):
    X = np.vstack([np.random.default_rng(1).standard_normal((70, 9)), np.zeros((3, 9))])   # zero rows: exact zeros
    with emulated_device() as lib:
        CV.check_sub_gram(CV.kernels()[kind], X, CV.ragged_rows(len(X), 3), layout)
        assert lib.emu_sticky_error() == 0


@pytest.mark.parametrize('sms,chunk', [(None, None), (2, 25), (5, 7)])
def test_svc_folds_equal_their_own_fits(monkeypatch, sms, chunk):
    if sms:
        monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', str(sms))
        monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', str(chunk))
    X, y = _binary()
    with emulated_device() as lib:
        est = SB.svc(CV.kernels()['gaussian'], tol=1e-3)
        ours, _ = CV.check_folds_equal_own_fits(est, X, y, CV.ragged_rows(len(X), 3), params=[{'C': 0.5}, {'C': 4.0}])
        assert CV.shared(ours) and {e.fit_times_['batch'] for e in ours} == {6}
        assert lib.emu_sticky_error() == 0


def test_a_fold_stopped_at_max_iter_next_to_finished_ones(monkeypatch):
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '3')
    monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', '16')
    X, y = _binary()
    rows = CV.ragged_rows(len(X), 3, seed=4)
    with emulated_device() as lib:
        free, _ = CV.check_folds_equal_own_fits(SB.svc(tol=1e-3), X, y, rows)
        iters = sorted(e.optimizer.iter for e in free)
        assert iters[0] < iters[-1]
        ours, _ = CV.check_folds_equal_own_fits(SB.svc(tol=1e-3, max_iter=iters[-1] - 1), X, y, rows)
        status = [e.optimizer.status for e in ours]
        assert 'stopped' in status and 'optimal' in status
        assert lib.emu_sticky_error() == 0


def test_svr_folds_equal_their_own_fits(monkeypatch):
    monkeypatch.setenv('SVMB200_SMO_BATCH_SMS', '4')
    monkeypatch.setenv('SVMB200_SMO_BATCH_CHUNK', '40')
    spec, X, y = make_config('C2', n=70)
    with emulated_device() as lib:
        ours, _ = CV.check_folds_equal_own_fits(SB.svr(tol=1e-4), X, y, CV.ragged_rows(len(X), 3, seed=2),
                                                params=[{'epsilon': 0.05}, {'epsilon': 0.2, 'C': 3.0}])
        assert CV.shared(ours)
        assert lib.emu_sticky_error() == 0


def test_grid_search_equals_sklearns():
    X, y = load_iris(return_X_y=True)
    X, y = X[y > 0], y[y > 0]
    with emulated_device() as lib:
        ours, _ = CV.grid_search_both(SB.svc(tol=1e-3), {'C': [0.1, 1.0, 10.0]}, X, y, cv=3, return_train_score=True)
        assert 'batch' not in ours.best_estimator_.fit_times_   # the refit is an ordinary single fit
        assert lib.emu_sticky_error() == 0


def test_grid_search_with_gamma_scale_builds_one_matrix_per_fold():
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.model_selection import _fit_and_score_shared
    from sklearn.metrics import check_scoring
    X, y = _binary(n=80)
    est = SB.svc(kernel=GaussianKernel(gamma='scale'), tol=1e-3)
    with emulated_device() as lib:
        CV.grid_search_both(est, [{'C': [0.5, 2.0]}, {'C': [1.0], 'kernel__gamma': [0.05, 'auto']}], X, y, cv=3,
                            scoring=['accuracy', 'balanced_accuracy'], refit='balanced_accuracy')
        splits = list(StratifiedKFold(3).split(X, y))
        out = _fit_and_score_shared(est, X, y, [{'C': 0.5}, {'C': 2.0}], splits, check_scoring(est), False, np.nan,
                                    return_estimator=True)
        fits = [o['estimator'] for o in out]
        # the two values of C share each fold's own matrix: one matrix per fold, two problems on each
        assert all(e.fit_times_['batch'] == 2 for e in fits)
        assert len({id(e.obj.device_hessian().matrix) for e in fits}) == 3
        assert lib.emu_sticky_error() == 0


def test_cross_validate_and_score_equal_sklearns():
    from sklearn.model_selection import cross_val_score as sklearn_cvs
    from optiml_b200.model_selection import cross_val_score
    spec, X, y = make_config('C2', n=60)
    with emulated_device() as lib:
        ours = CV.cross_validate_both(SB.svr(tol=1e-4), X, y, cv=KFold(4, shuffle=True, random_state=0),
                                      scoring=['r2', 'neg_mean_squared_error'], return_train_score=True,
                                      return_estimator=True, return_indices=True)
        assert CV.shared(ours['estimator'])
        Xc, yc = _binary(n=60)
        assert np.array_equal(cross_val_score(SB.svc(tol=1e-3), Xc, yc, cv=3),
                              sklearn_cvs(SB.svc(tol=1e-3), Xc, yc, cv=3))
        assert lib.emu_sticky_error() == 0


def test_fall_backs_keep_sklearns_results(monkeypatch, capsys):
    from optiml_b200.ml.svm import DualSVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge, squared_hinge
    X, y = _binary(n=60)
    with emulated_device() as lib:
        CV.grid_search_both(SB.svc(tol=1e-3, verbose=True), {'C': [1.0]}, X, y, cv=2, shared=False)
        capsys.readouterr()
        # fit parameters (SVC.fit's X_device), a projected-gradient estimator
        CV.grid_search_both(SB.svc(tol=1e-3), {'C': [1.0]}, X, y, cv=2, fit_params={'X_device': None}, shared=False)
        CV.grid_search_both(DualSVC(kernel=GaussianKernel(0.2), max_iter=50), {'C': [1.0, 2.0]}, X, y, cv=2,
                            shared=False)
        # a training fold with one class, and a candidate whose fit raises: sklearn's own handling
        y_one = y.copy()
        y_one[:30] = 1
        CV.grid_search_both(SB.svc(tol=1e-3), {'C': [1.0]}, X, y_one, cv=KFold(2), shared=False)
        ours, _ = CV.grid_search_both(SB.svc(tol=1e-3), {'loss': [hinge, squared_hinge]}, X, y, cv=2, shared=False)
        assert np.isnan(ours.cv_results_['mean_test_score'][1]) and ours.best_index_ == 0
        monkeypatch.setenv('SVMB200_SMO_ROWS', 'computed')   # M would not stay resident: clone after clone
        ours = CV.cross_validate_both(SB.svc(tol=1e-3), X, y, cv=3, return_estimator=True)
        assert not CV.shared(ours['estimator'])   # fit_shared_gram fitted the clones one after the other
        assert all(e.optimizer.row_source == 'computed' for e in ours['estimator'])
        assert lib.emu_sticky_error() == 0


def test_sharded_context_keeps_sklearns_not_implemented_error(monkeypatch):
    from optiml_b200 import runtime
    from optiml_b200.model_selection import GridSearchCV, cross_validate

    class ShardedContext:   # what default_context() is under torchrun with two ranks; any device call would fail
        nranks, group = 2, None
    monkeypatch.setattr(runtime, '_default_ctx', ShardedContext())
    X, y = _binary(n=40)
    with pytest.raises(NotImplementedError, match='one GPU'):
        GridSearchCV(SB.svc(), {'C': [1.0, 2.0]}, cv=2, error_score='raise').fit(X, y)
    with pytest.raises(NotImplementedError, match='one GPU'):
        cross_validate(SB.svc(), X, y, cv=2, error_score='raise')


def test_subset_abi_refusals():
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        X, y = _binary(n=40)
        est = SB.svc()
        H = est._build_hessian(X, None, 'plain', None, 0.0)
        est._train_X_device[0].release()
        n = H.n
        ys = np.where(y > 0, 1.0, -1.0)

        def create(active, ub=None, signs=ys):
            h = C.c_void_p()
            act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8)
            rc = lib.svmb200_smo_create_subset(ctx.handle, C.c_void_p(H.matrix.dptr), n, H.ld, 0, n, N.HESSIAN_PLAIN,
                                               N.ptr(signs), N.ptr(-np.ones(n)), N.ptr(np.ones(n) if ub is None else ub),
                                               None if act is None else act.ctypes.data_as(C.c_void_p), 1e-3, 100,
                                               C.byref(h))
            if rc == 0:
                lib.svmb200_pg_destroy(h)
            return rc, lib.svmb200_last_error()

        half = np.arange(n) < n // 2
        assert create(half)[0] == 0
        rc, err = create(ys > 0)
        assert rc == 1 and b'the active variables must hold both signs of the equality constraint' in err
        assert create(np.zeros(n))[0] == 1
        assert b'finite and > 0' in create(half, ub=np.where(half, 0.0, 1.0))[1]
        # an inactive variable's upper bound is not read: 0, a NaN or an infinity there is fine
        assert create(half, ub=np.where(half, 1.0, np.nan))[0] == 0
        assert create(half, ub=np.where(half, 1.0, 0.0))[0] == 0
        assert b'signs must be +-1' in create(half, signs=np.where(half, ys, 0.0))[1]
        assert create(None)[0] == 1
        # the plain creation keeps its check on every variable
        h = C.c_void_p()
        assert lib.svmb200_smo_create_signed(ctx.handle, C.c_void_p(H.matrix.dptr), n, H.ld, 0, n, N.HESSIAN_PLAIN,
                                             N.ptr(ys), N.ptr(-np.ones(n)), N.ptr(np.where(half, 1.0, 0.0)), 1e-3, 100,
                                             C.byref(h)) == 1
        assert b'upper bounds must be finite and > 0' in lib.svmb200_last_error()
        H.release()
        assert lib.emu_sticky_error() == 0


def test_a_subset_solver_runs_in_a_batch_with_plain_signed_views():
    with emulated_device() as lib:
        from optiml_b200.runtime import default_context
        ctx = default_context()
        X, y = _binary(n=60)
        est = SB.svc()
        H = est._build_hessian(X, None, 'plain', None, 0.0)
        est._train_X_device[0].release()
        n = H.n
        ys = np.where(y > 0, 1.0, -1.0)
        act = np.ascontiguousarray(np.arange(n) % 4 != 1, dtype=np.uint8)

        class Subset(SB.Problem):
            def __init__(self):
                self.h, self.nvars = C.c_void_p(), n
                N.call('svmb200_smo_create_subset', ctx.handle, C.c_void_p(H.matrix.dptr), n, H.ld, 0, n,
                       N.HESSIAN_PLAIN, N.ptr(ys), N.ptr(-np.ones(n)), N.ptr(np.ones(n)), act.ctypes.data_as(C.c_void_p),
                       1e-5, 10 ** 6, C.byref(self.h))

        SB.check_batch_equals_single_runs(lambda: [SB.Problem(ctx, H, ys, -np.ones(n), 1e-5, 10 ** 6), Subset()], lib)
        p = Subset()
        p.run()
        x = p.result()[0]
        p.destroy()
        assert np.all(x[act == 0] == 0) and np.any(x[act == 1] > 0)
        H.release()
        assert lib.emu_sticky_error() == 0


def test_search_returns_its_allocations():
    X, y = _binary(n=60)
    with emulated_device() as lib:
        base = lib.emu_live_allocations()
        from optiml_b200.model_selection import GridSearchCV
        from optiml_b200.runtime import default_context
        search = GridSearchCV(SB.svc(tol=1e-3), {'C': [0.5, 2.0]}, cv=3).fit(X, y)
        assert search.best_estimator_.optimizer.status == 'optimal'
        del search
        gc.collect()
        default_context().trim()
    assert lib.emu_live_allocations() == base   # the context is gone with everything the search allocated
