"""Several solvers on ONE resident matrix, advanced in lockstep on the GPU(s) (SURVEY.md 8f-4).

The reference has no such entry point: its users wrap ``SVC`` in sklearn's ``OneVsRestClassifier``
(ml/tests/test_svc.py:101-147), which clones the estimator per class; every clone rebuilds the same Gram matrix and
its solver streams its own ``Q = (y_c y_c') o (K + 1)`` three times per iteration.  The binary problems differ in the
label signs only, so here they share one unsigned ``M = K + bias`` in HBM (``DeviceHessian.with_signs``) and
``svmb200_pg_run_batch`` streams it once per iteration for up to four problems at a time.  Every solver ends with
exactly the state its own ``minimize()`` would have produced (the multi-vector pass reproduces the single-vector
reductions bit for bit), so this is a scheduling decision, not a different algorithm.

SMO solvers (ml/svm/smo.py) batch differently: an SMO iteration reads two rows and is bound by the latency of its grid
barriers, so ``svmb200_smo_run_batch`` runs the problems side by side on disjoint ranges of the GPU's SMs, each with its
own tol and max_iter, and each again ends bit for bit where its own ``minimize()`` would.
"""
import ctypes as C

from .. import _native as N
from ..runtime import KernelRowsHessian
from .constrained._device_loop import DeviceLoopMixin


def batchable(solvers):
    """True when ``minimize_batch`` can run the solvers together: device-resident solvers of one class on the same
    resident matrix, same iteration limit (SMO: each keeps its own), nothing to run on the host between iterations."""
    from ..ml.svm.smo import SMO
    solvers = list(solvers)
    if len(solvers) < 2:
        return False
    first = solvers[0]
    if not all(isinstance(s, DeviceLoopMixin) and type(s) is type(first) for s in solvers):
        return False
    if not all(s._resident_ok() and not getattr(s, 'profile', False) for s in solvers):
        return False
    if not isinstance(first, SMO) and len({int(s.max_iter) for s in solvers}) != 1:
        return False
    H0 = first.f.device_hessian()
    if isinstance(H0, KernelRowsHessian):
        return False   # SMO with computed rows has no batch
    if len(H0.shards()) != 1:
        return False   # a single-process device group advances one problem at a time (no lockstep batches there)
    for s in solvers:
        H = s.f.device_hessian()
        if H.matrix is not H0.matrix or H.layout != H0.layout or (H.row0, H.nrows) != (H0.row0, H0.nrows):
            return False
    return True


def minimize_batch(solvers):
    """``[s.minimize() for s in solvers]`` with the streaming passes shared.  Falls back to exactly that loop (still on
    the device, one solver after the other) when the solvers cannot advance in lockstep -- generic callbacks,
    ``verbose``, different matrices or solver classes."""
    from ..ml.svm.smo import SMO
    solvers = list(solvers)
    if not batchable(solvers):
        for s in solvers:
            s.minimize()
            s.batch_size_ = 1
        return solvers
    lib = N.load_library()
    created = []
    # a lockstep batch streams the matrix with the multi-vector FULL pass: its solvers are created with the symmetric
    # pass (runtime.use_symmetric_pass) switched off, so that their first product follows the same order as the rest
    ctxs = {}
    for s in solvers:
        c = getattr(s.f.device_hessian(), 'ctx', None)
        if c is not None and id(c) not in ctxs:
            was = C.c_int(0)
            N.call('svmb200_ctx_get_symmetric', c.handle, C.byref(was))
            ctxs[id(c)] = (c, was.value)
            N.call('svmb200_ctx_set_symmetric', c.handle, 0)
    try:
        try:
            for s in solvers:
                created.append(s._create(False))
        finally:
            for c, was in ctxs.values():
                N.call('svmb200_ctx_set_symmetric', c.handle, was)
        count = len(created)
        handles = (C.c_void_p * count)(*[h.value for h, _ in created])
        iters, statuses = (C.c_int64 * count)(), (C.c_int * count)()
        N.call('svmb200_smo_run_batch' if isinstance(solvers[0], SMO) else 'svmb200_pg_run_batch', handles, count, iters,
               statuses)
        for s, (h, n), it, st in zip(solvers, created, iters, statuses):
            s._finish_resident(h, n, int(it), N.STATUS[int(st)])
            s._after_run(h, n)       # device_ms / q_passes are those of the whole batch
            s.batch_size_ = count
    finally:
        for h, _ in created:
            lib.svmb200_pg_destroy(h)
    return solvers
