"""The exact symmetric pass (K2e, optiml_b200/csrc/k2_exact.cuh) on the B200: the default product of a one-GPU fit over a
self-Gram, read from the upper triangle with the full pass's bits.  The checks of tests/exact_symv_checks.py with the
shipped 8192-column segments, and the headline configuration under both settings of SVMB200_EXACT_SYMV against the
REAL reference's golden run.  (A sharded fit -- the full pass on every shard -- against the one-GPU fit, bit for bit, is
tests/test_gpu_multi.py; its C4 case has two segments, so its one-GPU side takes this pass.)
"""
import numpy as np
import pytest

import exact_symv_checks as EX
from shared_gram_checks import real_device
from optiml_b200.configs import make_config
from test_gpu_estimators import api, check_stable_fit

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('n', [8229, 17000])
def test_self_gram_is_exactly_symmetric(n):
    EX.check_self_gram_symmetry(real_device, n, 128, shards=((0, 4096), (4096, n - 4096)))


def test_self_gram_is_exactly_symmetric_at_c4():
    """n = 50 000, d = 128: every kernel, on the 3000 x 3000 submatrix of a seeded row sample (a 20 GB Gram is not brought
    to the host), and the Gaussian self-Gram's upper triangle against the cross-Gram's on those rows"""
    import ctypes as C
    from optiml_b200 import _native as N
    from optiml_b200.runtime import default_context
    n, d = 50000, 128
    X, _ = EX.data(n, d)
    rows = np.sort(np.random.default_rng(1).choice(n, 3000, replace=False))
    with real_device() as probe:
        ctx = default_context()
        dX = ctx.upload_matrix(X)
        ld = N.padded_ld(n)
        out = ctx.malloc(n * ld * 8)
        for kind in EX.KID:
            subs = []
            for same in (1, 0):
                gamma, coef0, degree = EX.PARAMS[kind]
                N.call('svmb200_gram', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, C.c_void_p(dX.dptr), n, dX.ld, d, same,
                       EX.KID[kind], gamma, coef0, degree, None, None, 0.0, 0, n, C.c_void_p(out), ld)
                S = np.empty((rows.size, rows.size))
                buf = np.empty(ld)
                for i, r in enumerate(rows):
                    ctx.d2h(buf, out + int(r) * ld * 8)
                    S[i] = buf[rows]
                subs.append(S)
                if kind != 'gaussian':
                    break
            assert np.array_equal(subs[0], subs[0].T), kind
            if kind == 'gaussian':
                iu = np.triu_indices(rows.size, 1)
                assert np.array_equal(subs[0][iu], subs[1][iu])
        ctx.free(out)
        dX.release()
        probe.assert_clean()


@pytest.mark.parametrize('n,kinds,signed', [(8229, tuple(EX.KID), False), (17000, ('gaussian', 'laplacian', 'poly'), True),
                                            (50000, ('gaussian',), True)])
def test_exact_product_equals_the_full_pass(n, kinds, signed):
    EX.check_exact_product(real_device, n, 128, 8192, kinds=kinds, signed=signed, poison=n < 50000)


def test_fits_are_bit_identical_with_and_without_the_exact_pass():
    EX.check_exact_fits(real_device, 9000, max_iter=60)


def test_c4_headline_bit_identical_under_both_settings(golden):
    """BASELINE headline config against the unmodified reference's 1000 iterations with the exact pass (the default) and
    with SVMB200_EXACT_SYMV=0: the same bits, and north_star's bar -- alpha within 1e-8, identical support set"""
    A = api()
    g = golden('c4_full_svc_gaussian')
    spec, X, y = make_config('C4')
    out = {}
    for on in (True, False):
        with EX.exact_symv(on):
            m = A['DualSVC'](kernel=A['GaussianKernel'](), C=1).fit(X, y)
        assert m.optimizer.exact_symv_pass is on
        out[on] = (m.alphas_.copy(), np.array(m.train_loss_history), float(m.intercept_))
        if on:
            check_stable_fit(m, g)
            assert len(m.support_) == 49020
        m.obj.release()
        del m
    assert np.array_equal(out[True][0], out[False][0]) and np.array_equal(out[True][1], out[False][1])
    assert out[True][2] == out[False][2]
