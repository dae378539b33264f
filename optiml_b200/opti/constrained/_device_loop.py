"""Shared host driver of the device-resident box-constrained QP solvers (ProjectedGradient, FrankWolfe).

Both reference solvers have the same outer shape (projected_gradient.py:76-143, frank_wolfe.py:88-165):
evaluate f, g and a direction, call the callback, test two stopping criteria, take an exact line-search
step.  On the device that is one streaming pass over Q plus one vector kernel per iteration
(csrc/pg.cu); this mixin only decides how often the host looks at the state.
"""
import ctypes as C

import numpy as np

from ... import _native as N


class GroupHandle(C.c_void_p):
    """Solver handles of the ranks of a single-process device group (runtime.DeviceGroup).  It IS the rank-0 handle
    wherever one handle is expected -- state, histories and statistics are replicated -- and carries its peers for the
    calls that drive all ranks: run and destroy."""
    peers = ()


def create_solvers(symbol, H, tail):
    """``symbol(ctx, shard, n, ld, row0, nrows, layout[, signs], *tail(h))`` for every shard of the resident matrix H:
    one handle under torchrun / on one GPU, one per rank (started together) on a single-process device group."""
    layout = N.HESSIAN_SVR if H.layout == 'svr' else N.HESSIAN_PLAIN
    handles = []
    try:
        for part in H.shards():
            h = C.c_void_p()
            head = (part.ctx.handle, C.c_void_p(part.matrix.dptr), part.n, part.ld, part.row0, part.nrows, layout)
            if H.signs is not None:
                # Q = (s s') o M on a shared, unsigned resident matrix (one-vs-rest, SURVEY.md 8f-4)
                N.call(symbol + '_signed', *head, N.ptr(H.signs), *tail(h))
            else:
                N.call(symbol, *head, *tail(h))
            handles.append(h)
            if getattr(part.matrix, 'self_gram', False):
                N.call('svmb200_pg_set_self_gram', h, 1)
        if len(handles) == 1:
            return handles[0]
        arr = (C.c_void_p * len(handles))(*[h.value for h in handles])
        N.call('svmb200_pg_start_group', arr, len(handles))
    except Exception:
        for h in handles:
            N.load_library().svmb200_pg_destroy(h)
        raise
    gh = GroupHandle(handles[0].value)
    gh.peers = tuple(handles)
    return gh


def destroy_solvers(h):
    lib = N.load_library()
    for peer in (getattr(h, 'peers', None) or (h,)):
        lib.svmb200_pg_destroy(peer)


class DeviceLoopMixin:
    # subclasses set these
    _create_symbol = None          # C entry point that builds the solver handle
    _verbose_header = ''

    def _extra_create_args(self):
        return ()

    def _print_iteration(self, scalars):
        raise NotImplementedError

    # ------------------------------------------------------------------ device solver handle
    def _create(self, profile=False):
        H = self.f.device_hessian()
        n = H.nvars
        if self.ub.size != n or self.lb.size != n or self.x.size != n:
            raise ValueError('bounds / start point size does not match with Q')
        q, lb, ub, x0 = (np.ascontiguousarray(v, dtype=np.float64) for v in (self.f.q, self.lb, self.ub, self.x))
        h = create_solvers(self._create_symbol, H,
                           lambda hh: (N.ptr(q), N.ptr(lb), N.ptr(ub), N.ptr(x0), float(self.eps), int(self.max_iter),
                                       *self._extra_create_args(), C.byref(hh)))
        self._after_create(h, profile)
        return h, n

    def _after_create(self, h, profile):
        """Profiling on request, and which pass the solver's products take (csrc/pg.cu, product_pass)."""
        if profile:
            N.call('svmb200_pg_set_profile', h, 1)
        on = C.c_int(0)
        N.call('svmb200_pg_is_symmetric', h, C.byref(on))
        self.symmetric_pass = bool(on.value)   # products from the upper triangle only (runtime.use_symmetric_pass)
        N.call('svmb200_pg_is_exact_symv', h, C.byref(on))
        self.exact_symv_pass = bool(on.value)   # the full pass's bits from the upper triangle (a self-Gram on one GPU)

    @staticmethod
    def _run(h, max_new):
        it, st = C.c_int64(0), C.c_int(0)
        peers = getattr(h, 'peers', None)
        if peers:
            arr = (C.c_void_p * len(peers))(*[p.value for p in peers])
            N.call('svmb200_pg_run_group', arr, len(peers), int(max_new), C.byref(it), C.byref(st))
        else:
            N.call('svmb200_pg_run', h, int(max_new), C.byref(it), C.byref(st))
        return int(it.value), N.STATUS[st.value]

    def _pull_state(self, h, n):
        x, g = np.empty(n), np.empty(n)
        f, ng = C.c_double(0), C.c_double(0)
        N.call('svmb200_pg_state', h, N.ptr(x), N.ptr(g), C.byref(f), C.byref(ng))
        self.x, self.g_x, self.f_x = x, g, float(f.value)
        return float(ng.value)

    @staticmethod
    def _scalars(h):
        vals = np.zeros(6)
        N.call('svmb200_pg_scalars', h, N.ptr(vals))
        return vals

    def _history_only_callback(self):
        """True when nothing has to run on the host between iterations: no callback, or the estimators' own
        ``_store_train_info`` (ml/svm/_base.py:289-293) which only appends f_x."""
        cb = self._callback
        return cb is None or getattr(cb, '_svmb200_history_only', False) or \
            getattr(getattr(cb, '__func__', None), '_svmb200_history_only', False)

    def _problem_ndim(self):
        return self.f.ndim

    def _resident_ok(self):
        """The whole loop can stay on the device: nothing runs on the host between iterations."""
        return self._history_only_callback() and not self.verbose and self._problem_ndim() > 3

    def minimize(self):
        if self.verbose:
            print(self._verbose_header, end='')
        profile = bool(getattr(self, 'profile', False))
        h, n = self._create(profile)
        try:
            if self._resident_ok():
                self._minimize_resident(h, n)
            else:
                self._minimize_stepwise(h, n)
            self._after_run(h, n)
        finally:
            destroy_solvers(h)
        if self.verbose:
            print('\n')
        return self

    def _after_run(self, h, n):
        self._collect_stats(h)

    def _minimize_resident(self, h, n):
        # whole loop on the device; f at every callback point comes back in one copy
        self._finish_resident(h, n, *self._run(h, -1))

    def _finish_resident(self, h, n, it, status):
        """Collect the outcome of a device-resident run (also used by the batched driver, opti/batch.py)."""
        self.iter, self.status = it, status
        self._pull_state(h, n)
        cnt = C.c_int64(0)
        f_hist, second = np.empty(self.iter + 1), np.empty(self.iter + 1)
        N.call('svmb200_pg_history', h, N.ptr(f_hist), N.ptr(second), C.byref(cnt))
        self.f_hist, self.ng_hist = f_hist[:cnt.value], second[:cnt.value]
        if self._callback is not None and not self._extend_owner_history(self.f_hist):
            # replay the history-only callback: one call per callback point, in order
            final_f, final_iter = self.f_x, self.iter
            for k, fk in enumerate(self.f_hist):
                self.iter, self.f_x = k, float(fk)
                self._callback(self, *self.callback_args)
            self.iter, self.f_x = final_iter, final_f

    def _extend_owner_history(self, values):
        """The estimators' own callback (ml/svm/_base.py:289-293) appends one number per callback point to
        ``train_loss_history``; when that is the callback, the 1001 Python calls of a replay are one ``list.extend``."""
        cb = self._callback
        owner = getattr(cb, '__self__', None)
        if owner is None or not getattr(getattr(cb, '__func__', None), '_svmb200_history_only', False) or self.callback_args:
            return False
        hist = getattr(owner, 'train_loss_history', None)
        if not isinstance(hist, list):
            return False
        hist.extend(np.asarray(values, dtype=np.float64).tolist())
        return True

    def _minimize_stepwise(self, h, n):
        # generic callbacks / verbose / ndim <= 3 histories: synchronise at every callback point
        self.iter, status = self._run(h, 0)
        while True:
            self._pull_state(h, n)
            if self.is_verbose():
                self._print_iteration(self._scalars(h))
            try:
                self.callback()
            except StopIteration:
                break
            if status != 'unknown':
                self.status = status
                break
            self.iter, status = self._run(h, 1)

    def _collect_stats(self, h):
        ms, passes, mv = C.c_float(0), C.c_int64(0), C.c_float(0)
        N.call('svmb200_pg_stats', h, C.byref(ms), C.byref(passes), C.byref(mv))
        self.device_ms, self.q_passes, self.matvec_ms = float(ms.value), int(passes.value), float(mv.value)
        cm, vm = C.c_float(0), C.c_float(0)
        N.call('svmb200_pg_stats_ex', h, C.byref(mv), C.byref(cm), C.byref(vm))
        self.comm_ms, self.vector_ms = float(cm.value), float(vm.value)
        ns = C.c_int64(0)
        N.call('svmb200_pg_profile_samples', h, C.byref(ns))
        self.profile_samples = int(ns.value)   # iterations that carried CUDA events (one in 16 with profiling on)
