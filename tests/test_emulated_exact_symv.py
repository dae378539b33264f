"""The exact symmetric pass (K2e) and the exact symmetry of K1's self-Grams on the host emulation, with column segments
of 512 and 1024 instead of 8192 so that small problems have several of them (the checks: tests/exact_symv_checks.py;
the same run on the B200 in tests/test_gpu_exact_symv.py)."""
import pytest

import exact_symv_checks as EX
from test_emulated_kernels import emu_probe

# segment width, rows per sub-block, copies per batch, ring depth (a chain of K2 has 2 * segment / 512 rows)
_SEG512 = ('SVMB200_MV_SEG=512', 'SVMB200_EXACT_TR=2', 'SVMB200_EXACT_LB=1', 'SVMB200_EXACT_STAGES=2')
_SEG1024 = ('SVMB200_MV_SEG=1024', 'SVMB200_EXACT_TR=2', 'SVMB200_EXACT_LB=1', 'SVMB200_EXACT_STAGES=3')
_SEG1024_TR4 = ('SVMB200_MV_SEG=1024', 'SVMB200_EXACT_TR=4', 'SVMB200_EXACT_LB=2', 'SVMB200_EXACT_STAGES=2')


@pytest.mark.parametrize('n,d', [(130, 5), (203, 17), (333, 40)])
def test_self_gram_is_exactly_symmetric(n, d):
    EX.check_self_gram_symmetry(emu_probe, n, d, shards=((0, 64), (64, 64), (128, n - 128)))


@pytest.mark.parametrize('n,defines,seg', [(1030, _SEG512, 512), (1536, _SEG512, 512), (1100, _SEG1024, 1024),
                                           (2300, _SEG1024_TR4, 1024)])
def test_exact_product_equals_the_full_pass(n, defines, seg):
    kinds = ('gaussian', 'laplacian', 'poly') if n == 1030 else ('gaussian',)
    EX.check_exact_product(emu_probe, n, 6, seg, kinds=kinds, defines=defines)


@pytest.mark.parametrize('order,seed', [(1, 1), (2, 5)])
def test_exact_product_signed_layout_and_schedules(order, seed):
    w0 = EX.check_exact_product(emu_probe, 1100, 6, 512, signed=True, defines=_SEG512)
    w1 = EX.check_exact_product(emu_probe, 1100, 6, 512, signed=True, poison=False, defines=_SEG512, order=order, seed=seed)
    assert all((a == b).all() for a, b in zip(w0, w1))


def test_fits_are_bit_identical_with_and_without_the_exact_pass():
    EX.check_exact_fits(emu_probe, 600, max_iter=15, defines=_SEG512)


def test_exact_pass_applies_only_where_it_is_exact(monkeypatch):
    """one segment, a user-supplied matrix, the opt-in symmetric pass, a sharded matrix or SMO: the full pass; the
    augmented-Lagrangian solvers take the exact pass like the box-constrained ones"""
    import ctypes as C
    import numpy as np
    from optiml_b200 import _native as N, runtime
    from optiml_b200.ml.svm import SVC, DualSVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge
    from optiml_b200.opti import Quadratic
    from optiml_b200.opti.constrained import ProjectedGradient
    from optiml_b200.opti.unconstrained.stochastic import AdaGrad
    from symv_checks import symmetric_pass
    X, y = EX.data(600, 4)
    with emu_probe(defines=_SEG512), EX.exact_symv(True):
        m = DualSVC(kernel=GaussianKernel(), max_iter=3).fit(X[:400], y[:400])
        assert not m.optimizer.exact_symv_pass   # 400 < 512: one segment
        m.obj.release()
        with symmetric_pass(True):
            m = DualSVC(kernel=GaussianKernel(), max_iter=3).fit(X, y)
            assert m.optimizer.symmetric_pass and not m.optimizer.exact_symv_pass
            m.obj.release()
        m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, reg_intercept=False, dual=True, optimizer=AdaGrad, learning_rate=1.,
                max_iter=3, random_state=5).fit(X, y)
        assert m.optimizer.exact_symv_pass
        m.obj.release()
        Q = np.eye(600) + 0.01
        pg = ProjectedGradient(quad=Quadratic(Q, np.ones(600)), ub=np.ones(600), max_iter=3).minimize()
        assert not pg.exact_symv_pass
        pg.f.release()
        # SMO takes no products: svmb200_pg_set_self_gram leaves it alone
        ctx = runtime.default_context()
        ld = 608
        Qp = np.zeros((600, ld))
        Qp[:, :600] = Q
        dQ = ctx.malloc(Qp.nbytes)
        ctx.h2d(dQ, Qp)
        ones = np.ones(600)
        h, on = C.c_void_p(), C.c_int(1)
        N.call('svmb200_smo_create', ctx.handle, C.c_void_p(dQ), 600, ld, 0, 600, N.HESSIAN_PLAIN, N.ptr(ones), N.ptr(-ones),
               N.ptr(ones), 1e-3, 10, C.byref(h))
        try:
            N.call('svmb200_pg_set_self_gram', h, 1)
            N.call('svmb200_pg_is_exact_symv', h, C.byref(on))
            assert on.value == 0
        finally:
            N.load_library().svmb200_pg_destroy(h)
            ctx.free(dQ)
        # a matrix sharded over a single-process group of two GPUs
        monkeypatch.setattr(runtime.DeviceGroup, 'MIN_ROWS_PER_GPU', 64)
        runtime.use_devices([0, 1])
        try:
            m = DualSVC(kernel=GaussianKernel(), max_iter=3).fit(X, y)
            assert len(m.obj.device_hessian().shards()) == 2 and not m.optimizer.exact_symv_pass
            m.obj.release()
        finally:
            runtime.use_devices(None)
