"""Creation and teardown of the solver handle (csrc/pg.cu) on the host emulation: every allocation a solver makes is
returned when it is destroyed, or when its creation is refused part-way, and no write strays outside its buffer (the
emulation's canaries around every allocation are checked when it is freed)."""
import ctypes as C

import numpy as np

from emu import emulated_device
from optiml_b200 import _native as N
from optiml_b200.runtime import Context, DeviceGroup, DeviceHessian


def _problem(n, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, 3))
    y = np.where(X[:, 0] + 0.5 * rng.standard_normal(n) > 0, 1.0, -1.0)
    return X, y, -np.ones(n), np.ones(n)


def _run(h, max_new):
    it, status = C.c_int64(), C.c_int()
    N.call('svmb200_pg_run', h, max_new, C.byref(it), C.byref(status))
    return it.value


def _close(lib, base, ctxs, *buffers):
    for b in buffers:
        b.release()
    for c in ctxs:
        c.trim()
        c._finalizer()
    assert lib.emu_live_allocations() == base
    assert lib.emu_sticky_error() == 0


def test_resident_smo_fit_returns_its_allocations():
    X, y, q, ub = _problem(70, 1)
    Q = (y[:, None] * y[None, :]) * np.exp(-((X[:, None] - X[None]) ** 2).sum(-1) / 3)
    with emulated_device() as lib:
        base = lib.emu_live_allocations()
        ctx = Context(device=0)
        H = DeviceHessian.from_host(ctx, Q)
        live = None
        for _ in range(2):   # the first fit also takes the context's grid barrier, which stays with the context
            h = C.c_void_p()
            N.call('svmb200_smo_create', ctx.handle, C.c_void_p(H.matrix.dptr), 70, H.ld, 0, 70, N.HESSIAN_PLAIN,
                   N.ptr(y), N.ptr(q), N.ptr(ub), 1e-3, 10 ** 5, C.byref(h))
            assert _run(h, -1) > 0
            N.call('svmb200_pg_destroy', h)
            assert live is None or lib.emu_live_allocations() == live
            live = lib.emu_live_allocations()
        _close(lib, base, [ctx], H)


def test_computed_row_smo_with_a_regrown_history_returns_its_allocations():
    n = 60
    X, y, q, ub = _problem(n, 4)
    with emulated_device() as lib:
        base = lib.emu_live_allocations()
        ctx = Context(device=0)
        dX = ctx.upload_matrix(X)
        h = C.c_void_p()
        # gaussian (row norms in the row buffer), a two-row cache, tol = 0: the solve keeps going
        N.call('svmb200_smo_create_rows', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, 3, 2, 1 / 3, 0.0, 3.0,
               N.HESSIAN_PLAIN, N.ptr(y), N.ptr(q), N.ptr(np.full(n, 100.0)), 0.0, 10 ** 6, 2 * n * 8, C.byref(h))
        assert _run(h, 600) == 600 and _run(h, 600) == 1200
        count, slots = C.c_int64(), C.c_int64()
        N.call('svmb200_pg_history', h, None, None, C.byref(count))
        N.call('svmb200_smo_cache_stats', h, None, C.byref(slots), None, None)
        assert count.value == 1201 and slots.value == 2   # the history grew past its first 1 024 states
        N.call('svmb200_pg_destroy', h)
        _close(lib, base, [ctx], dX)


def test_two_live_solvers_on_one_context_destroyed_in_either_order():
    n = 40
    X, y, q, ub = _problem(n, 2)
    with emulated_device() as lib:
        base = lib.emu_live_allocations()
        ctx = Context(device=0)
        H = DeviceHessian.from_host(ctx, X @ X.T + np.eye(n))

        def create():
            h = C.c_void_p()
            N.call('svmb200_pg_create', ctx.handle, C.c_void_p(H.matrix.dptr), n, H.ld, 0, n, N.HESSIAN_PLAIN, N.ptr(q),
                   None, N.ptr(ub), None, 1e-9, 50, C.byref(h))
            _run(h, 20)
            return h

        N.call('svmb200_pg_destroy', create())   # the context's workspace and scratch, kept for later solves
        idle = lib.emu_live_allocations()
        for order in ((0, 1), (1, 0)):
            pair = [create()]
            shared = lib.emu_live_allocations()
            pair.append(create())
            assert shared == idle and lib.emu_live_allocations() == idle + 2   # the second: private slab + pinned block
            for i in order:
                N.call('svmb200_pg_destroy', pair[i])
            assert lib.emu_live_allocations() == idle
        _close(lib, base, [ctx], H)


def test_creation_refused_after_it_has_allocated():
    """a single-process group whose last rank owns no rows: creation takes the context's workspace, then finds that the
    fused exchange is impossible, and must give the workspace back"""
    n = 100   # three ranks of 64-row shards: rank 2 owns nothing
    X, y, q, ub = _problem(n, 3)
    with emulated_device() as lib:
        base = lib.emu_live_allocations()
        group = DeviceGroup([0, 1, 2])
        ctx = group.ctxs[0]
        H = DeviceHessian(ctx, n)
        assert (H.row0, H.nrows) == (0, 64)
        live = []
        for _ in range(2):
            h = C.c_void_p()
            rc = lib.svmb200_pg_create(ctx.handle, C.c_void_p(H.matrix.dptr), n, H.ld, H.row0, H.nrows, N.HESSIAN_PLAIN,
                                       N.ptr(q), None, N.ptr(ub), None, 1e-6, 10, C.byref(h))
            assert rc == 1 and not h.value   # SVMB200_ERR_ARG
            assert b'a single-process group needs the fused exchange' in lib.svmb200_last_error()
            live.append(lib.emu_live_allocations())
        assert live[1] == live[0]   # the second attempt found the workspace free again: no private one
        _close(lib, base, group.ctxs, H)
