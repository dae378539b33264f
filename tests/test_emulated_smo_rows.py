"""K12 (computed rows for K11: csrc/kernel_fn.cuh, the ROWS = computed instantiation of csrc/k_smo.cuh) executed on the
host emulation of the CUDA runtime (tests/cuda_emu): the kernel values against the oracle's kernels and against K1, fits
without a resident Hessian bit-identical to oracle/smo_oracle.py replayed on the matrix assembled from
svmb200_kernel_rows, the same bits for every cache size, schedule and call pattern, and the choice of the row source."""
import ctypes as C

import numpy as np
import pytest

from emu import emulated_device
from oracle import smo_oracle as SO
from oracle import svm_oracle as O
from optiml_b200.configs import make_config

KERNELS = ['linear', 'poly', 'gaussian', 'sigmoid', 'laplacian']
KID = {'linear': 0, 'poly': 1, 'gaussian': 2, 'sigmoid': 3, 'laplacian': 4}


def _device_rows(X, kind, gamma, coef0, degree, rows):
    """(svmb200_kernel_rows, svmb200_gram) on the emulated device: the listed rows of K from both"""
    from optiml_b200 import _native as N
    from optiml_b200.runtime import DeviceMatrix, default_context
    ctx = default_context()
    n, d = X.shape
    dX = ctx.upload_matrix(X)
    ld = N.padded_ld(n)
    rows = np.ascontiguousarray(rows, dtype=np.int64)
    out = DeviceMatrix(ctx, len(rows), n, ld)
    N.call('svmb200_kernel_rows', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, d, KID[kind], gamma, coef0, degree,
           rows.ctypes.data_as(C.c_void_p), len(rows), C.c_void_p(out.dptr), ld)
    K = DeviceMatrix(ctx, n, n, ld)
    N.call('svmb200_gram', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, C.c_void_p(dX.dptr), n, dX.ld, d, 1, KID[kind],
           gamma, coef0, degree, None, None, 0.0, 0, n, C.c_void_p(K.dptr), ld)
    ctx.sync()
    return out.to_host(), K.to_host()[rows]


@pytest.mark.parametrize('kind', KERNELS)
@pytest.mark.parametrize('n,d', [(70, 1), (65, 7), (40, 10), (33, 37)])
def test_kernel_rows_equal_k1_and_the_oracle(kind, n, d):
    rng = np.random.default_rng(n * 100 + d)
    X = rng.standard_normal((n, d)) * 0.7
    gamma, coef0, degree = 1.0 / d, 0.5, 3
    rows = [0, n - 1, n // 2, 3, 3]
    with emulated_device() as lib:
        got, k1 = _device_rows(X, kind, gamma, coef0, degree, rows)
        assert lib.emu_sticky_error() == 0
    assert np.array_equal(got, k1)   # K1's order on the emulation: bit for bit
    want = O.kernel_matrix(kind, X, degree=degree, gamma=gamma, coef0=coef0)[rows]
    np.testing.assert_allclose(got, want, rtol=1e-13, atol=1e-13 * np.abs(want).max())


def test_non_integer_degree_takes_pow_as_k1_does():
    X = np.random.default_rng(3).standard_normal((30, 5))
    with emulated_device():
        got, k1 = _device_rows(X, 'poly', 0.3, 2.0, 2.5, [1, 7])
    assert np.array_equal(got, k1, equal_nan=True)   # a negative base has no real power: NaN in both


def fit(monkeypatch, task, n, grid=3, kernel='gaussian', cache_mb=None, order=0, tol=1e-5, max_iter=10 ** 6,
        callback=None):
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm import kernels as Kn
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    monkeypatch.setenv('SVMB200_SMO_GRID', str(grid))
    monkeypatch.setenv('SVMB200_SMO_ROWS', 'computed')
    if cache_mb is None:
        monkeypatch.delenv('SVMB200_SMO_CACHE_MB', raising=False)
    else:
        monkeypatch.setenv('SVMB200_SMO_CACHE_MB', repr(cache_mb))
    k = {'gaussian': Kn.GaussianKernel(), 'poly': Kn.PolyKernel(degree=3), 'linear': Kn.LinearKernel(),
         'laplacian': Kn.LaplacianKernel()}[kernel]
    if task == 'svc':
        spec, X, y = make_config('C1', n=n)
        m = SVC(loss=hinge, kernel=k, C=1, dual=True, optimizer='smo', tol=tol, max_iter=max_iter)
    else:
        spec, X, y = make_config('C2', n=n)
        m = SVR(loss=epsilon_insensitive, kernel=k, C=1, epsilon=0.1, dual=True, optimizer='smo', tol=tol,
                max_iter=max_iter)
    with emulated_device(order=order, seed=5) as lib:
        m.fit(X, y)
        Q = m.obj.device_hessian().to_host()
        assert lib.emu_sticky_error() == 0
    return m, Q


def outcome(o):
    return o.x, o.g_x, o.f_hist, o.gap_hist, o.iter, o.status, o.rho


def assert_same(a, b):
    for u, v in zip(outcome(a), outcome(b)):
        assert np.array_equal(u, v)


@pytest.mark.parametrize('task,n,kernel', [('svc', 131, 'gaussian'), ('svc', 257, 'gaussian'), ('svr', 97, 'poly'),
                                           ('svc', 131, 'linear'), ('svc', 131, 'laplacian')])
@pytest.mark.parametrize('grid', [1, 3, 8])
def test_computed_fit_is_bit_identical_to_the_oracle(monkeypatch, task, n, kernel, grid):
    m, Q = fit(monkeypatch, task, n, grid, kernel)
    o = m.optimizer
    assert o.row_source == 'computed'
    r = SO.smo(Q, o.f.q, o.y, o.ub, tol=1e-5, max_iter=10 ** 6)
    assert o.status == r.status == 'optimal' and o.iter == r.iter
    for got, want in ((o.x, r.x), (o.g_x, r.g), (o.f_hist, r.f_hist), (o.gap_hist, r.gap_hist)):
        assert np.array_equal(got, want)
    assert o.rho == r.rho and m.intercept_ == -r.rho


def test_computed_rows_equal_the_resident_fit(monkeypatch):
    """K12 follows K1's order, so on the emulation the computed Hessian is K1's and the two fits agree bit for bit"""
    m, Q = fit(monkeypatch, 'svc', 131)
    monkeypatch.setenv('SVMB200_SMO_ROWS', 'resident')
    from optiml_b200.ml.svm import SVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge
    spec, X, y = make_config('C1', n=131)
    r = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=1e-5, max_iter=10 ** 6)
    with emulated_device():
        r.fit(X, y)
        assert np.array_equal(r.obj.device_hessian().to_host(), Q)
    assert r.optimizer.row_source == 'resident'
    assert_same(m.optimizer, r.optimizer)
    assert np.array_equal(m.support_, r.support_) and np.array_equal(m.dual_coef_, r.dual_coef_)


def _touched_rows(Q, o, n):
    """the sample indices of every row the solver reads: row i of each evaluated state, row j of each step"""
    touched = set()
    y, C = o.y, o.ub
    for k in range(o.iter + 1):
        r = SO.smo(Q, o.f.q, y, C, tol=1e-5, max_iter=k)
        G, a = r.g, r.x
        up = np.where(y > 0, a < C, a > 0)
        i = SO._last_argmax(-(y * G), up)
        if i < 0:
            break
        touched.add(i % n)
        if k < o.iter:
            low = np.where(y > 0, a > 0, a < C)
            b = -(y[i] * G[i]) + y * G
            at = (Q[i, i] + np.diagonal(Q)) - (2.0 * y[i] * y) * Q[i]
            at = np.where(at <= 0, SO.TAU, at)
            with np.errstate(divide='ignore', invalid='ignore'):
                j = SO._last_argmax((b * b) / at, low & (b > 0))
            touched.add(j % n)
    return touched


def test_cache_size_never_changes_a_bit(monkeypatch):
    n = 60
    runs = {}
    for slots in (0, 1, 2, 5, n):
        runs[slots], Q = fit(monkeypatch, 'svc', n, 3, cache_mb=slots * n * 8 / (1 << 20))
    base = runs[0].optimizer
    assert base.cache_slots == 0 and base.cache_hits == 0
    for slots, m in runs.items():
        o = m.optimizer
        assert o.cache_slots == slots
        assert_same(o, base)
        assert o.cache_hits + o.cache_misses == base.cache_misses   # the same lookups, whatever the cache holds
    full = runs[n].optimizer
    assert full.cache_misses == len(_touched_rows(Q, full, n))    # one miss per distinct row
    assert runs[1].optimizer.cache_hits <= runs[5].optimizer.cache_hits


def test_svr_rows_share_a_slot(monkeypatch):
    """SVR rows s and s + n are the same samples: a cache of all n rows never misses twice on one sample"""
    n = 40
    m, Q = fit(monkeypatch, 'svr', n, 3, kernel='poly', cache_mb=n * 2 * n * 8 / (1 << 20))
    o = m.optimizer
    assert o.cache_slots == n and o.cache_misses <= n
    r = SO.smo(Q, o.f.q, o.y, o.ub, tol=1e-5, max_iter=10 ** 6)
    assert np.array_equal(o.x, r.x) and o.iter == r.iter


@pytest.mark.parametrize('order', [1, 2])
def test_thread_and_block_schedules_do_not_change_a_bit(monkeypatch, order):
    a, _ = fit(monkeypatch, 'svc', 131, 8, cache_mb=0.05)
    b, _ = fit(monkeypatch, 'svc', 131, 8, cache_mb=0.05, order=order)
    assert_same(a.optimizer, b.optimizer)
    assert (a.optimizer.cache_hits, a.optimizer.cache_misses) == (b.optimizer.cache_hits, b.optimizer.cache_misses)


def test_one_iteration_calls_equal_one_run(monkeypatch):
    from optiml_b200.ml.svm.smo import SMO
    from optiml_b200.opti import Quadratic
    from optiml_b200.runtime import KernelRowsHessian, default_context
    m, Q = fit(monkeypatch, 'svc', 131, 3, cache_mb=0.05)
    spec, X, y = make_config('C1', n=131)
    seen = []
    with emulated_device() as lib:
        ctx = default_context()
        H = KernelRowsHessian(ctx, ctx.upload_matrix(X), X, (KID['gaussian'], m.kernel.gram_spec(X)[1], 0., 3.),
                              'plain', m.optimizer.y, cache_bytes=5 * 131 * 8)
        o = SMO(quad=Quadratic(H, m.optimizer.f.q), y=m.optimizer.y, C=1., tol=1e-5, max_iter=10 ** 6,
                callback=lambda opt: seen.append(opt.iter)).minimize()
        assert lib.emu_sticky_error() == 0
        H.release()
    assert seen == list(range(o.iter + 1))
    assert o.row_source == 'computed' and o.cache_slots == 5
    assert_same(o, m.optimizer)


def test_product_of_the_computed_hessian(monkeypatch):
    from optiml_b200.runtime import KernelRowsHessian, default_context
    spec, X, y = make_config('C2', n=50)
    v = np.random.default_rng(0).standard_normal(100)
    with emulated_device():
        ctx = default_context()
        H = KernelRowsHessian(ctx, ctx.upload_matrix(X), X, (KID['poly'], 0.1, 1.0, 3.0), 'svr')
        Q = H.to_host()
        got = H.product(v)
        H.release()
    np.testing.assert_allclose(got, Q @ v, rtol=1e-10, atol=1e-10 * np.abs(Q @ v).max())


class TestRowSource:
    INFO = dict(sm_count=148, free_bytes=180 << 30)

    def select(self, n, svr=False, d=64, **info):
        from optiml_b200 import _native as N
        from optiml_b200.ml.svm.smo import select_row_source
        nvars = 2 * n if svr else n
        with emulated_device():
            return select_row_source(n, nvars, N.padded_ld(n), d, dict(self.INFO, **info))

    def test_resident_while_the_matrix_fits(self, monkeypatch):
        monkeypatch.delenv('SVMB200_SMO_ROWS', raising=False)
        monkeypatch.delenv('SVMB200_SMO_CACHE_MB', raising=False)
        assert self.select(50_000) == ('resident', 0)
        assert self.select(1000, free_bytes=9 << 20) == ('resident', 0)

    def test_computed_beyond_free_memory_with_a_bounded_cache(self, monkeypatch):
        monkeypatch.delenv('SVMB200_SMO_ROWS', raising=False)
        monkeypatch.delenv('SVMB200_SMO_CACHE_MB', raising=False)
        n = 200_000
        src, cache = self.select(n)
        assert src == 'computed'
        assert 0 < cache <= 0.8 * (180 << 30) and cache % (n * 8) == 0
        src, cache = self.select(1000, free_bytes=7 << 20)   # 8 MB matrix, 7 MB free: all 1000 rows still fit the cache
        assert src == 'computed' and cache <= 1000 * 1000 * 8

    def test_overrides(self, monkeypatch):
        monkeypatch.setenv('SVMB200_SMO_ROWS', 'computed')
        monkeypatch.setenv('SVMB200_SMO_CACHE_MB', '1')
        assert self.select(1000) == ('computed', (1 << 20) // 8000 * 8000)
        monkeypatch.setenv('SVMB200_SMO_ROWS', 'resident')
        assert self.select(300_000) == ('resident', 0)
        monkeypatch.setenv('SVMB200_SMO_ROWS', 'sideways')
        with pytest.raises(ValueError):
            self.select(1000)

    def test_size_limit(self, monkeypatch):
        monkeypatch.delenv('SVMB200_SMO_ROWS', raising=False)
        assert self.select(697_672)[0] == 'computed'
        assert self.select(348_836, svr=True)[0] == 'computed'
        with pytest.raises(ValueError, match='697672'):
            self.select(697_673)
        with pytest.raises(ValueError, match='697672'):
            self.select(348_837, svr=True)

    def test_estimator_refuses_before_any_device_work(self, monkeypatch):
        from optiml_b200.ml.svm import SVC
        from optiml_b200.ml.svm.losses import hinge
        monkeypatch.setenv('SVMB200_SMO_ROWS', 'computed')
        X = np.zeros((700_000, 1))
        y = np.where(np.arange(700_000) % 2 == 0, 1.0, -1.0)
        with emulated_device() as lib:
            import optiml_b200.runtime as R
            ctx = R.default_context()
            monkeypatch.setattr(type(ctx), 'info', lambda self: dict(TestRowSource.INFO))
            before = lib.emu_launches()
            with pytest.raises(ValueError, match='697672'):
                SVC(loss=hinge, C=1, dual=True, optimizer='smo').fit(X, y)
            assert lib.emu_launches() == before


def test_integration_md_smo_rows_stub_runs_against_the_emulated_library():
    """the ctypes stub `smo_rows` of INTEGRATION.md, executed, against the oracle on the rows the library computes"""
    import os
    import re
    import emu
    from optiml_b200.runtime import KernelRowsHessian, default_context
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, 'INTEGRATION.md')) as fh:
        blocks = re.findall(r'```python\n(.*?)```', fh.read(), flags=re.S)
    ns = {}
    exec(compile('\n'.join(blocks).replace("'libsvmb200.so'", repr(emu._builder().build())), 'INTEGRATION.md', 'exec'), ns)
    rng = np.random.default_rng(2)
    X = rng.standard_normal((90, 6))
    y = np.where(rng.integers(0, 2, 90) == 1, 1., -1.)
    gamma = 1.0 / 6
    a, g, it, status = ns['smo_rows'](X, -np.ones(90), y, kernel=KID['gaussian'], gamma=gamma, tol=1e-5,
                                      cache_bytes=7 * 90 * 8)
    with emulated_device():
        ctx = default_context()
        H = KernelRowsHessian(ctx, ctx.upload_matrix(X), X, (KID['gaussian'], gamma, 0., 3.), 'plain', y)
        Q = H.to_host()
        H.release()
    want = SO.smo(Q, -np.ones(90), y, 1., tol=1e-5)
    assert it == want.iter and status == want.status == 'optimal'
    assert np.array_equal(a, want.x) and np.array_equal(g, want.g)
