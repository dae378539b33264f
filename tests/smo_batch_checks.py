"""Shared checks of SMO on signed views of one unsigned M and of the SMO batch (csrc/k_smo.cuh K14,
``svmb200_smo_run_batch``, ml/multiclass.py): the CPU suite runs them on the host emulation, the GPU suite on the B200."""
import ctypes as C
import warnings

import numpy as np
from sklearn.exceptions import ConvergenceWarning

from optiml_b200 import _native as N


def svc(kernel=None, **kw):
    from optiml_b200.ml.svm import SVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge
    return SVC(loss=hinge, kernel=kernel or GaussianKernel(), C=1, dual=True, optimizer='smo', **kw)


def svr(**kw):
    from optiml_b200.ml.svm import SVR
    from optiml_b200.ml.svm.kernels import PolyKernel
    from optiml_b200.ml.svm.losses import epsilon_insensitive
    return SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo', **kw)


def quantile_classes(X, k, seed=0):
    """multi-class labels on any inputs: quantiles of a fixed random projection (scripts/bench_ovr.py)"""
    score = X @ np.random.default_rng(seed).standard_normal(X.shape[1])
    return np.searchsorted(np.quantile(score, np.linspace(0, 1, k + 1)[1:-1]), score)


def outcome(o):
    return o.x, o.g_x, o.f_hist, o.gap_hist, o.iter, o.status


def assert_same_solve(a, b):
    for u, v in zip(outcome(a), outcome(b)):
        assert np.array_equal(u, v)


# ------------------------------------------------------------------ signed views
def signed_view_against_k1(est, X, ys, tol=1e-5, max_iter=10 ** 6):
    """SMO on K1's signed Q against SMO on the signed view of K1's unsigned M (both bias 0); returns the two solvers
    and K1's signed Q on the host"""
    from optiml_b200.ml.svm.smo import SMO
    from optiml_b200.opti import Quadratic
    from optiml_b200.runtime import default_context
    n = len(ys)
    q, ub = -np.ones(n), np.ones(n)
    dX = default_context().upload_matrix(X)
    Hq = est._build_hessian(X, ys, 'plain', dX, 0.0)
    Hm = est._build_hessian(X, None, 'plain', dX, 0.0)
    dX.release()
    try:
        a = SMO(quad=Quadratic(Hq, q), y=ys, C=ub, tol=tol, max_iter=max_iter).minimize()
        b = SMO(quad=Quadratic(Hm.with_signs(ys), q), y=ys, C=ub, tol=tol, max_iter=max_iter).minimize()
        Q = Hq.to_host()
    finally:
        Hq.release()
        Hm.release()
    return a, b, Q


# ------------------------------------------------------------------ the C ABI of the batch
class Problem:
    """one SMO problem on the shared M of `ctx`: create it (by default a resident SVR problem or a signed SVC view),
    run it alone or in a batch, read its outcome"""

    def __init__(self, ctx, H, sign, q, tol, max_iter, svr=False, signed=None):
        self.h = C.c_void_p()
        layout = N.HESSIAN_SVR if svr else N.HESSIAN_PLAIN
        signed = not svr if signed is None else signed
        symbol = 'svmb200_smo_create_signed' if signed else 'svmb200_smo_create'
        self.nvars = len(q)
        N.call(symbol, ctx.handle, C.c_void_p(H.matrix.dptr), H.n, H.ld, 0, H.n, layout, N.ptr(sign), N.ptr(q),
               N.ptr(np.ones(self.nvars)), float(tol), int(max_iter), C.byref(self.h))

    def run(self):
        it, st = C.c_int64(), C.c_int()
        N.call('svmb200_pg_run', self.h, -1, C.byref(it), C.byref(st))
        return it.value, st.value

    def result(self):
        x, g = np.empty(self.nvars), np.empty(self.nvars)
        f, gap, cnt = C.c_double(), C.c_double(), C.c_int64()
        N.call('svmb200_pg_state', self.h, N.ptr(x), N.ptr(g), C.byref(f), C.byref(gap))
        N.call('svmb200_pg_history', self.h, None, None, C.byref(cnt))
        fh, gh = np.empty(cnt.value), np.empty(cnt.value)
        N.call('svmb200_pg_history', self.h, N.ptr(fh), N.ptr(gh), C.byref(cnt))
        return x, g, f.value, gap.value, fh, gh

    def destroy(self):
        N.load_library().svmb200_pg_destroy(self.h)


def run_batch(problems, lib=None):
    lib = lib or N.load_library()
    arr = (C.c_void_p * len(problems))(*[p.h.value for p in problems])
    iters, sts = (C.c_int64 * len(problems))(), (C.c_int * len(problems))()
    rc = lib.svmb200_smo_run_batch(arr, len(problems), iters, sts)
    return rc, list(iters), list(sts)


def batch_problems(ctx, H, X, count, svr_targets=None, max_iters=None, tol=1e-5):
    """`count` problems on H: signed one-vs-rest views of quantile classes of X, or SVR targets"""
    n = H.n
    out = []
    for b in range(count):
        mi = (max_iters or {}).get(b, 10 ** 6)
        if svr_targets is not None:
            y = svr_targets[:, b]
            out.append(Problem(ctx, H, np.hstack((np.ones(n), -np.ones(n))), np.hstack((-y, y)) + 0.1, tol, mi, svr=True))
        else:
            labels = quantile_classes(X, max(count, 2), seed=b // 2)
            ys = np.where(labels == b % max(count, 2), 1.0, -1.0)
            out.append(Problem(ctx, H, ys, -np.ones(n), tol * (1 + b % 3), mi))
    return out


def check_batch_equals_single_runs(make_problems, lib=None):
    """make_problems() -> fresh problems on one M; the batch must end where every problem's own run ends, bit for bit"""
    alone = make_problems()
    want = []
    for p in alone:
        it, st = p.run()
        want.append((it, st) + p.result())
        p.destroy()
    together = make_problems()
    try:
        rc, iters, sts = run_batch(together, lib)
        assert rc == 0, N.load_library().svmb200_last_error()
        for p, it, st, w in zip(together, iters, sts, want):
            got = (it, st) + p.result()
            assert got[:2] == w[:2]
            for u, v in zip(got[2:], w[2:]):
                assert np.array_equal(u, v)
    finally:
        for p in together:
            p.destroy()
    return want


# ------------------------------------------------------------------ estimators
def compare_estimators(ours, theirs, X):
    assert len(ours) == len(theirs)
    for a, b in zip(ours, theirs):
        for u, v in ((a.alphas_, b.alphas_), (a.support_, b.support_), (a.dual_coef_, b.dual_coef_)):
            assert np.array_equal(u, v)
        assert a.intercept_ == b.intercept_
        oa, ob = a.optimizer, b.optimizer
        assert oa.iter == ob.iter and oa.status == ob.status and np.array_equal(oa.f_hist, ob.f_hist)


def compare_ovr(est, X, y):
    """our OneVsRestClassifier (one M, SMO batch) against sklearn's clone-per-class fit: bitwise; returns ours"""
    from sklearn.multiclass import OneVsRestClassifier as SklearnOVR
    from optiml_b200.ml.multiclass import OneVsRestClassifier
    with warnings.catch_warnings(record=True) as w_ours:
        warnings.simplefilter('always')
        ours = OneVsRestClassifier(est).fit(X, y)
    with warnings.catch_warnings(record=True) as w_sk:
        warnings.simplefilter('always')
        theirs = SklearnOVR(est).fit(X, y)
    compare_estimators(ours.estimators_, theirs.estimators_, X)
    assert np.array_equal(ours.decision_function(X), theirs.decision_function(X))
    assert np.array_equal(ours.predict(X), theirs.predict(X))
    conv = [sum(issubclass(x.category, ConvergenceWarning) for x in w) for w in (w_ours, w_sk)]
    assert conv[0] == conv[1]
    return ours, theirs


def assert_one_shared_matrix(estimators):
    Ms = {id(e.obj.device_hessian().matrix) for e in estimators}
    assert len(Ms) == 1
    assert all(e.fit_times_.get('batch') == len(estimators) for e in estimators)
