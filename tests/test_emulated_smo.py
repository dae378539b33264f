"""K11 (csrc/k_smo.cuh, the SMO solver) executed on the host emulation of the CUDA runtime (tests/cuda_emu): whole
estimator fits are bit-identical to oracle/smo_oracle.py replayed on the matrix the kernel read, for grids of 1, 3 and
8 CTAs, under other thread and block schedules, and when the run is chopped into one-iteration calls."""
import warnings

import numpy as np
import pytest
from sklearn.exceptions import ConvergenceWarning

from emu import emulated_device
from oracle import smo_oracle as SO
from optiml_b200.configs import make_config


def fit(monkeypatch, task, n, grid, order=0, max_iter=10 ** 6, tol=1e-5):
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    monkeypatch.setenv('SVMB200_SMO_GRID', str(grid))
    if task == 'svc':
        spec, X, y = make_config('C1', n=n)
        m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=max_iter)
    else:
        spec, X, y = make_config('C2', n=n)
        m = SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo',
                tol=tol, max_iter=max_iter)
    with emulated_device(order=order, seed=5) as lib:
        m.fit(X, y)
        Q = m.obj.device_hessian().to_host()
        assert lib.emu_sticky_error() == 0
    return m, Q


def outcome(o):
    return o.x, o.g_x, o.f_hist, o.gap_hist, o.iter, o.status


def assert_same(a, b):
    for u, v in zip(outcome(a), outcome(b)):
        assert np.array_equal(u, v)


@pytest.mark.parametrize('task,n', [('svc', 131), ('svc', 257), ('svr', 97)])
@pytest.mark.parametrize('grid', [1, 3, 8])
def test_estimator_fit_is_bit_identical_to_the_oracle(monkeypatch, task, n, grid):
    m, Q = fit(monkeypatch, task, n, grid)
    o = m.optimizer
    r = SO.smo(Q, o.f.q, o.y, o.ub, tol=1e-5, max_iter=10 ** 6)
    assert o.status == r.status == 'optimal'
    assert o.iter == r.iter
    for got, want in ((o.x, r.x), (o.g_x, r.g), (o.f_hist, r.f_hist), (o.gap_hist, r.gap_hist)):
        assert np.array_equal(got, want)
    assert o.rho == r.rho and o.f_x == r.f_x and m.intercept_ == -r.rho
    assert o.gap == r.gap_hist[-1] < 1e-5


@pytest.mark.parametrize('order', [1, 2])
def test_thread_and_block_schedules_do_not_change_a_bit(monkeypatch, order):
    a, _ = fit(monkeypatch, 'svc', 131, 8)
    b, _ = fit(monkeypatch, 'svc', 131, 8, order=order)
    assert_same(a.optimizer, b.optimizer)


def test_one_iteration_calls_equal_one_run(monkeypatch):
    """a generic callback makes the solver synchronise at every state: svmb200_pg_run(h, 1) per iteration"""
    from optiml_b200.opti import Quadratic
    from optiml_b200.ml.svm.smo import SMO
    m, Q = fit(monkeypatch, 'svc', 131, 3)
    seen = []
    with emulated_device() as lib:
        o = SMO(quad=Quadratic(Q, m.optimizer.f.q), y=m.optimizer.y, C=1., tol=1e-5, max_iter=10 ** 6,
                callback=lambda opt: seen.append(opt.iter)).minimize()
        assert lib.emu_sticky_error() == 0
    assert seen == list(range(o.iter + 1))
    assert_same(o, m.optimizer)


def test_max_iter_stops_with_a_convergence_warning(monkeypatch):
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        m, Q = fit(monkeypatch, 'svr', 97, 3, max_iter=25)
    assert any(issubclass(x.category, ConvergenceWarning) for x in w)
    o = m.optimizer
    assert o.status == 'stopped' and o.iter == 25 and len(o.f_hist) == 26
    r = SO.smo(Q, o.f.q, o.y, o.ub, tol=1e-5, max_iter=25)
    assert r.status == 'stopped' and np.array_equal(o.x, r.x) and np.array_equal(o.gap_hist, r.gap_hist)


def test_integration_md_smo_stub_runs_against_the_emulated_library():
    """the ctypes stub `smo` of INTEGRATION.md, executed, against the oracle"""
    import os
    import re
    import emu
    from oracle import svm_oracle as O
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, 'INTEGRATION.md')) as fh:
        blocks = re.findall(r'```python\n(.*?)```', fh.read(), flags=re.S)
    ns = {}
    exec(compile('\n'.join(blocks).replace("'libsvmb200.so'", repr(emu._builder().build())), 'INTEGRATION.md', 'exec'), ns)
    rng = np.random.default_rng(1)
    X = rng.standard_normal((90, 6))
    y = np.where(rng.integers(0, 2, 90) == 1, 1., -1.)
    Q = y[:, None] * O.gaussian_kernel(X) * y[None, :]
    a, g, f_hist, gap_hist, it, status = ns['smo'](Q, -np.ones(90), y, tol=1e-5)
    want = SO.smo(Q, -np.ones(90), y, 1., tol=1e-5)
    assert it == want.iter and status == want.status == 'optimal'
    assert np.array_equal(a, want.x) and np.array_equal(g, want.g) and np.array_equal(f_hist, want.f_hist)
