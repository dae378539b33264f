"""Checks of the exact symmetric pass (K2e, optiml_b200/csrc/k2_exact.cuh: the full pass's product, bit for bit, from the
upper triangle of a self-Gram) and of the exact symmetry of K1's self-Grams it relies on.  Written once and run twice: on
the host emulation in the CPU suite (tests/test_emulated_exact_symv.py, built with small column segments,
-DSVMB200_MV_SEG=...) and on the B200 in the `-m gpu` suite (tests/test_gpu_exact_symv.py, the shipped 8192).

``device`` is a callable returning a context manager that yields a probe with ``launches()`` and ``assert_clean()``
(tests/shared_gram_checks.py).
"""
import contextlib
import ctypes as C
import os

import numpy as np

from optiml_b200 import _native as N

KID = {'linear': 0, 'poly': 1, 'gaussian': 2, 'sigmoid': 3, 'laplacian': 4}
PARAMS = {'linear': (0.0, 0.0, 3.0), 'poly': (0.3, 1.0, 3.0), 'gaussian': (0.2, 0.0, 3.0), 'sigmoid': (0.05, 0.1, 3.0),
          'laplacian': (0.1, 0.0, 3.0)}


@contextlib.contextmanager
def exact_symv(on):
    """SVMB200_EXACT_SYMV=0/1 for the solvers created inside the block"""
    saved = os.environ.get('SVMB200_EXACT_SYMV')
    os.environ['SVMB200_EXACT_SYMV'] = '1' if on else '0'
    try:
        yield
    finally:
        if saved is None:
            del os.environ['SVMB200_EXACT_SYMV']
        else:
            os.environ['SVMB200_EXACT_SYMV'] = saved


def data(n, d, seed=0):
    rng = np.random.default_rng(seed + n)
    X = rng.standard_normal((n, d))
    X[rng.integers(0, n, max(1, n // 50))] *= 3.0   # a few rows with larger norms
    return X, np.where(rng.standard_normal(n) >= 0, 1.0, -1.0)


def gram(ctx, dX, n, d, kind, same=1, signs=None, row0=0, nrows=None, bias=0.0):
    """rows [row0, row0 + nrows) of K1's n x n Gram of X with itself (same = 1: self-Gram) on the device, to the host"""
    nrows = n - row0 if nrows is None else nrows
    ld = N.padded_ld(n)
    out = ctx.malloc(max(nrows, 1) * ld * 8)
    dS = ctx.upload_vector(signs) if signs is not None else None
    sp = C.c_void_p(dS.dptr) if dS is not None else None
    gamma, coef0, degree = PARAMS[kind]
    N.call('svmb200_gram', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, C.c_void_p(dX.dptr), n, dX.ld, d, int(same), KID[kind],
           gamma, coef0, degree, sp, sp, float(bias), row0, nrows, C.c_void_p(out), ld)
    M = np.empty((max(nrows, 1), ld))
    ctx.d2h(M, out)
    ctx.free(out)
    if dS is not None:
        dS.release()
    return M[:nrows]


def check_self_gram_symmetry(device, n, d, kinds=tuple(KID), shards=(), **dev_kw):
    """K1's self-Gram equals its transpose bit for bit for every kernel; its upper triangle is the arithmetic of the
    cross-Gram (same = 0: sklearn's order everywhere), and row shards give the rows of the whole"""
    from optiml_b200.runtime import default_context
    X, _ = data(n, d)
    iu = np.triu_indices(n, 1)
    with device(**dev_kw) as probe:
        ctx = default_context()
        dX = ctx.upload_matrix(X)
        for kind in kinds:
            Q = gram(ctx, dX, n, d, kind)[:, :n]
            assert np.array_equal(Q, Q.T), kind
            cross = gram(ctx, dX, n, d, kind, same=0)[:, :n]
            assert np.array_equal(Q[iu], cross[iu]), kind
            for row0, nrows in shards:
                assert np.array_equal(gram(ctx, dX, n, d, kind, row0=row0, nrows=nrows)[:, :n], Q[row0:row0 + nrows]), kind
        dX.release()
        probe.assert_clean()


def _product(ctx, symbol, dQ, n, ld, u):
    du, dw = ctx.malloc(8 * ld), ctx.malloc(8 * n)
    ctx.h2d(du, u)
    ctx.memset(dw, 0xFF, 8 * n)
    N.call(symbol, ctx.handle, C.c_void_p(dQ), n, ld, C.c_void_p(du), C.c_void_p(dw))
    w = np.empty(n)
    ctx.d2h(w, dw)
    ctx.free(du)
    ctx.free(dw)
    return w


def check_exact_product(device, n, d, seg, kinds=('gaussian',), signed=False, poison=True, data_seed=0, **dev_kw):
    """svmb200_matvec_exact == svmb200_matvec bit for bit on K1 self-Grams (``signed``: with label signs, the layout of
    the SVC Hessian); with every block strictly below the seg x seg diagonal blocks NaN, the same bits again.  Returns
    the products."""
    from optiml_b200.runtime import default_context
    X, s = data(n, d, data_seed)
    ld = N.padded_ld(n)
    rng = np.random.default_rng(data_seed + 7)
    u = np.zeros(ld)
    u[:n] = rng.standard_normal(n) * (rng.random(n) < 0.7)   # zeros as in a projected direction
    out = []
    with device(**dev_kw) as probe:
        ctx = default_context()
        dX = ctx.upload_matrix(X)
        for kind in kinds:
            Q = gram(ctx, dX, n, d, kind, signs=s if signed else None, bias=1.0 if signed else 0.0)
            dQ = ctx.malloc(Q.nbytes)
            ctx.h2d(dQ, Q)
            w_full = _product(ctx, 'svmb200_matvec', dQ, n, ld, u)
            w_exact = _product(ctx, 'svmb200_matvec_exact', dQ, n, ld, u)
            assert np.array_equal(w_full, w_exact), kind
            assert np.abs(w_full - Q[:, :n] @ u[:n]).max() <= 1e-12 * n * max(1.0, np.abs(w_full).max())
            if poison:
                cols = np.arange(Q.shape[1])[None, :]
                Qp = Q.copy()
                Qp[(cols // seg < np.arange(n)[:, None] // seg) & (cols < n)] = np.nan
                ctx.h2d(dQ, Qp)
                assert np.array_equal(_product(ctx, 'svmb200_matvec_exact', dQ, n, ld, u), w_full), kind
            ctx.free(dQ)
            out.append(w_full)
        dX.release()
        probe.assert_clean()
    return out


def check_exact_fits(device, n, max_iter=20, **dev_kw):
    """DualSVC with projected gradient (plain layout and the label-sign view) and Frank-Wolfe, DualSVR (block layout):
    the same bits with SVMB200_EXACT_SYMV=0 (full pass) and =1 (exact symmetric pass), which the solvers report"""
    from optiml_b200.ml.svm import DualSVC, DualSVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, LaplacianKernel
    from optiml_b200.opti.constrained import FrankWolfe
    from sklearn.datasets import make_classification, make_regression
    X, y = make_classification(n_samples=n, n_features=8, random_state=3)
    Xr, yr = make_regression(n_samples=n, n_features=5, noise=0.1, random_state=4)
    yr = (yr - yr.mean()) / yr.std()
    out = {}
    for on in (False, True):
        with device(**dev_kw) as probe, exact_symv(on):
            pg = DualSVC(kernel=GaussianKernel(), max_iter=max_iter)
            pg.profile_matvec = True   # the two-kernel loop at any size (no persistent kernel)
            pg.fit(X, y)
            fw = DualSVC(kernel=LaplacianKernel(), optimizer=FrankWolfe, max_iter=max_iter).fit(X, y)
            svr = DualSVR(kernel=GaussianKernel(), max_iter=max_iter, epsilon=0.1)
            svr.profile_matvec = True
            svr.fit(Xr, yr)
            for m in (pg, fw, svr):
                assert m.optimizer.exact_symv_pass is on
            out[on] = [pg.alphas_.copy(), np.asarray(pg.train_loss_history).copy(), fw.alphas_.copy(), svr.alphas_.copy()]
            for m in (pg, fw, svr):
                m.obj.release()
            del pg, fw, svr
            probe.assert_clean()
    for a, b in zip(out[False], out[True]):
        assert np.array_equal(a, b)
    return out[True]
