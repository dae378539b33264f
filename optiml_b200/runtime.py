"""Device runtime of the host mirror: contexts (GPU + stream), device-resident matrices and the multi-GPU plumbing.

Two multi-GPU models, same kernels, same row-block partition, bit-identical results:

* one process per GPU (``torchrun``): ``torch.distributed`` is used only for the rendezvous (NCCL unique id, IPC handles of
  the exchange arenas); the per-iteration exchange is fused into the matvec kernel over NVLink peer memory, with an
  ``ncclAllGather`` issued by the C library as the fallback (csrc/comm.cu);
* ONE process, N GPUs (``use_devices([...])`` or ``SVMB200_DEVICES=0,1,...|all``): the reference's API is a single Python
  process calling ``SVC.fit``; a :class:`DeviceGroup` makes that process drive every GPU from the calling thread -- no
  torchrun, no torch, no NCCL -- so notebooks and sklearn meta-estimators (``GridSearchCV``) use all GPUs unchanged.
"""
import ctypes as C
import os
import weakref

import numpy as np

from . import _native as N

_default_ctx = None


class Context:
    """Owns a ``svmb200_ctx`` (one GPU, one stream)."""

    def __init__(self, device=None):
        if device is None:
            device = int(os.environ.get('LOCAL_RANK', '0'))
        count = C.c_int(0)
        N.call('svmb200_device_count', C.byref(count))
        h = C.c_void_p()
        N.call('svmb200_ctx_create', int(device) % max(count.value, 1), C.byref(h))
        self.handle = h
        self.device = int(device)
        self.rank, self.nranks = 0, 1
        self.group = None   # a DeviceGroup whose GPUs this (solo) context may fan large problems out to
        # large device buffers (the Hessian shard) are recycled between fits: cudaMalloc/cudaFree of
        # tens of GB costs ~0.1 s each, more than the Gram build itself
        self._pool = []  # (nbytes, device pointer), oldest first
        if _symmetric is not None:
            N.call('svmb200_ctx_set_symmetric', h, int(_symmetric))
        self._finalizer = weakref.finalize(self, N.load_library().svmb200_ctx_destroy, h)

    # ---------------------------------------------------------------- memory
    POOL_MIN_BYTES = 1 << 20
    POOL_MAX_BUFFERS = 4
    POOL_SLACK = 1.5   # parked bytes never exceed this multiple of the largest parked buffer (one Hessian shard + X)

    def malloc(self, nbytes):
        nbytes = int(nbytes)
        for i in range(len(self._pool) - 1, -1, -1):
            if self._pool[i][0] == nbytes:
                return self._pool.pop(i)[1]
        p = C.c_void_p()
        try:
            N.call('svmb200_malloc', self.handle, nbytes, C.byref(p))
        except N.NativeError:
            if not self._pool:
                raise
            self.trim()  # parked buffers of other sizes (earlier fits) may be what is in the way: give them back, retry once
            N.call('svmb200_malloc', self.handle, nbytes, C.byref(p))
        return p.value

    def free(self, dptr, nbytes=0):
        """Buffers of >= 1 MB are parked for the next fit of the same size (exact-size reuse): at most four, and never more
        bytes in total than 1.5x the largest parked one -- fits of varying n (CV folds, other data sets) evict the oldest
        parked buffers instead of accumulating Hessian-sized ones."""
        if not dptr:
            return
        nbytes = int(nbytes)
        if nbytes < self.POOL_MIN_BYTES:
            N.call('svmb200_free', self.handle, C.c_void_p(dptr))
            return
        self._pool.append((nbytes, dptr))
        while len(self._pool) > self.POOL_MAX_BUFFERS or \
                sum(sz for sz, _ in self._pool) > self.POOL_SLACK * max(sz for sz, _ in self._pool):
            _, victim = self._pool.pop(0)  # oldest first
            N.call('svmb200_free', self.handle, C.c_void_p(victim))

    def pooled_bytes(self):
        return sum(sz for sz, _ in self._pool)

    def trim(self):
        """Return pooled buffers to the driver."""
        pool, self._pool = self._pool, []
        for _, dptr in pool:
            N.call('svmb200_free', self.handle, C.c_void_p(dptr))

    def memset(self, dptr, value, nbytes):
        N.call('svmb200_memset', self.handle, C.c_void_p(dptr), int(value), int(nbytes))

    def h2d(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        N.call('svmb200_h2d', self.handle, C.c_void_p(dptr), arr.ctypes.data_as(C.c_void_p), arr.nbytes)

    def d2h(self, arr, dptr):
        assert arr.flags['C_CONTIGUOUS']
        N.call('svmb200_d2h', self.handle, arr.ctypes.data_as(C.c_void_p), C.c_void_p(dptr), arr.nbytes)

    def sync(self):
        N.call('svmb200_sync', self.handle)

    def timer_start(self):
        N.call('svmb200_timer_start', self.handle)

    def timer_stop_ms(self):
        ms = C.c_float(0)
        N.call('svmb200_timer_stop_ms', self.handle, C.byref(ms))
        return float(ms.value)

    def launch_count(self):
        """kernels launched through this context (and, for a solo context with a device group, through the group's)"""
        n = C.c_uint64(0)
        N.call('svmb200_launch_count', self.handle, C.byref(n))
        total = int(n.value)
        if self.group is not None:
            total += sum(c.launch_count() for c in self.group.ctxs)
        return total

    def info(self):
        sm, ma, mi = C.c_int(0), C.c_int(0), C.c_int(0)
        fr, to = C.c_size_t(0), C.c_size_t(0)
        N.call('svmb200_ctx_info', self.handle, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(fr), C.byref(to))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), free_bytes=fr.value, total_bytes=to.value)

    # ---------------------------------------------------------------- multi-GPU
    def attach_communicator(self, rank, nranks, unique_id):
        """Join the NCCL communicator described by ``unique_id`` (128 bytes from rank 0)."""
        buf = C.create_string_buffer(bytes(unique_id), 128)
        N.call('svmb200_comm_init', self.handle, C.cast(buf, C.c_void_p), int(rank), int(nranks))
        self.rank, self.nranks = int(rank), int(nranks)

    def enable_peer_exchange(self, dist, arena_bytes=64 << 20):
        """Map every rank's exchange arena (CUDA IPC over NVLink) so that the matvec kernel can store its
        shard straight into all peers.  Falls back to the NCCL all-gather if any rank cannot map."""
        buf = C.create_string_buffer(64)
        ok = True
        try:
            N.call('svmb200_comm_p2p_export', self.handle, int(arena_bytes), C.cast(buf, C.c_void_p))
        except N.NativeError:
            ok = False
        handles = [None] * self.nranks
        dist.all_gather_object(handles, buf.raw if ok else None)
        if any(h is None for h in handles):
            N.call('svmb200_comm_p2p_disable', self.handle)
            return False
        blob = C.create_string_buffer(b''.join(handles), 64 * self.nranks)
        try:
            N.call('svmb200_comm_p2p_attach', self.handle, C.cast(blob, C.c_void_p), self.nranks)
        except N.NativeError:
            ok = False
        flags = [None] * self.nranks
        dist.all_gather_object(flags, ok)
        self.peer_exchange = all(flags)
        if not self.peer_exchange:
            N.call('svmb200_comm_p2p_disable', self.handle)  # every rank must take the same path
        return self.peer_exchange

    @property
    def exchange(self):
        if self.nranks == 1:
            return 'none'
        en = C.c_int(0)
        N.call('svmb200_comm_p2p_enabled', self.handle, C.byref(en))
        return 'p2p' if en.value else 'nccl'

    @staticmethod
    def new_unique_id():
        buf = C.create_string_buffer(128)
        N.call('svmb200_comm_unique_id', C.cast(buf, C.c_void_p))
        return buf.raw

    def broadcast_array(self, arr, src=0):
        """Every rank gets rank ``src``'s copy of a host array (replicated solver inputs that were drawn at random
        must be identical on all ranks: the vector phase runs redundantly on each of them)."""
        if self.nranks == 1:
            return arr
        import torch.distributed as dist
        box = [arr if self.rank == src else None]
        dist.broadcast_object_list(box, src=src)
        return box[0]

    def row_shard(self, n):
        """Rows [row0, row0+nrows) of an n-row matrix owned by this rank."""
        return shard_rows(n, self.rank, self.nranks)

    # ---------------------------------------------------------------- matrices
    def upload_matrix(self, X):
        """Copy a host matrix to the device with an even leading dimension (16-byte row stride)."""
        X = np.ascontiguousarray(X, dtype=np.float64)
        n, d = X.shape
        ld = d + (d & 1)
        if ld != d:
            Xp = np.zeros((n, ld))
            Xp[:, :d] = X
            X = Xp
        m = DeviceMatrix(self, n, d, ld)
        self.h2d(m.dptr, X)
        return m

    def upload_vector(self, v, length=None):
        v = np.ascontiguousarray(v, dtype=np.float64).ravel()
        length = len(v) if length is None else int(length)
        out = DeviceMatrix(self, 1, length, max(length, 2))
        self.memset(out.dptr, 0, out.nbytes)
        self.h2d(out.dptr, v)
        return out


def shard_rows(n, rank, nranks):
    """(row0, nrows) of rank's shard: the partition of svmb200_shard_rows (single source of truth)."""
    r0, nr = C.c_int64(0), C.c_int64(0)
    N.call('svmb200_shard_rows', int(n), int(rank), int(nranks), C.byref(r0), C.byref(nr))
    return int(r0.value), int(nr.value)


class DeviceMatrix:
    """A row-major FP64 matrix in HBM (rows x cols, leading dimension ld)."""

    def __init__(self, ctx, rows, cols, ld):
        self.ctx, self.rows, self.cols, self.ld = ctx, int(rows), int(cols), int(ld)
        self.nbytes = max(self.rows, 1) * self.ld * 8
        self.dptr = ctx.malloc(self.nbytes)
        # rows of a self-Gram svmb200_gram built (same = 1): exactly symmetric, so a solver on one GPU may take its
        # products from the upper triangle with the full pass's bits (svmb200_pg_set_self_gram)
        self.self_gram = False
        self._finalizer = weakref.finalize(self, _free_quiet, ctx, self.dptr, self.nbytes)

    def release(self):
        self._finalizer()
        self.dptr = None

    def to_host(self):
        buf = np.empty((self.rows, self.ld))
        self.ctx.d2h(buf, self.dptr)
        return np.ascontiguousarray(buf[:, :self.cols])


def _free_quiet(ctx, dptr, nbytes=0):
    try:
        ctx.free(dptr, nbytes)
    except Exception:  # interpreter shutdown / context already gone
        pass


class DeviceHessian:
    """Row shard [row0, row0+nrows) of the n x n matrix the solver streams every iteration.

    ``layout='plain'``: the matrix is Q itself.  ``layout='svr'``: the matrix is M = K + 1 and the
    Hessian is [[M, -M], [-M, M]] (ml/svm/_base.py:1098-1099, 1178 of the reference) -- the 2n x 2n
    matrix is never materialised on the device.

    ``signs`` (n values of +-1, plain layout only): the resident matrix is M and the Hessian is
    Q = (s s') o M -- what ml/svm/_base.py:554, 628 build from the labels.  ``with_signs`` returns such a view
    of an unsigned matrix without copying it, so the binary problems of a one-vs-rest fit share one M in HBM
    (SURVEY.md 8f-4); the solvers apply s to their vectors, which is exact.
    """

    def __init__(self, ctx, n, layout='plain', matrix=None, row0=None, nrows=None, signs=None):
        self.ctx, self.n, self.layout = ctx, int(n), layout
        if row0 is None:
            row0, nrows = ctx.row_shard(n)
        self.row0, self.nrows = int(row0), int(nrows)
        self.ld = N.padded_ld(n)
        self.owns_matrix = matrix is None
        self.matrix = matrix if matrix is not None else DeviceMatrix(ctx, self.nrows, self.n, self.ld)
        self.signs = None
        if signs is not None:
            signs = np.ascontiguousarray(signs, dtype=np.float64).ravel()
            if layout != 'plain':
                raise ValueError('label signs apply to the plain layout only')
            if signs.size != self.n or not np.all(np.abs(signs) == 1.0):
                raise ValueError('signs must be n values of +-1')
            self.signs = signs

    def with_signs(self, signs):
        """A view of the same resident matrix whose Hessian is (s s') o M (no copy; the view does not own M)."""
        if self.signs is not None:
            raise ValueError('the matrix already carries label signs')
        return DeviceHessian(self.ctx, self.n, self.layout, matrix=self.matrix, row0=self.row0, nrows=self.nrows,
                             signs=signs)

    @property
    def nvars(self):
        return 2 * self.n if self.layout == 'svr' else self.n

    def shards(self):
        """the per-context shards a solver is created on (one here; a GroupHessian has one per rank)"""
        return [self]

    @classmethod
    def from_host(cls, ctx, Q):
        """Upload (this rank's rows of) a host-resident square matrix."""
        Q = np.asarray(Q, dtype=np.float64)
        n = Q.shape[0]
        h = cls(ctx, n, 'plain')
        block = np.zeros((max(h.nrows, 1), h.ld))
        block[:h.nrows, :n] = Q[h.row0:h.row0 + h.nrows]
        ctx.h2d(h.matrix.dptr, block)
        return h

    def shard_to_host(self):
        buf = np.empty((max(self.nrows, 1), self.ld))
        self.ctx.d2h(buf, self.matrix.dptr)
        return np.ascontiguousarray(buf[:self.nrows, :self.n])

    def to_host(self):
        """Materialise the full Hessian on the host (debug / parity / API compatibility only)."""
        M = self.shard_to_host()
        if self.ctx.nranks > 1:
            import torch.distributed as dist
            parts = [None] * self.ctx.nranks
            dist.all_gather_object(parts, M)
            M = np.vstack(parts)
        if self.layout == 'svr':
            return np.vstack((np.hstack((M, -M)), np.hstack((-M, M))))
        if self.signs is not None:
            return self.signs[:, None] * M * self.signs[None, :]
        return M

    def product(self, v):
        """Q @ v through the streaming matvec kernel (all ranks get the full result)."""
        v = np.asarray(v, dtype=np.float64).ravel()
        if self.layout == 'svr':
            beta = v[:self.n] - v[self.n:]
        elif self.signs is not None:
            beta = self.signs * v
        else:
            beta = v
        beta = np.ascontiguousarray(beta)
        out = np.empty(self.n)
        N.call('svmb200_masked_product', self.ctx.handle, C.c_void_p(self.matrix.dptr), self.n, self.ld, self.row0,
               self.nrows, N.ptr(beta), N.ptr(out))
        if self.signs is not None:
            out *= self.signs
        return np.concatenate((out, -out)) if self.layout == 'svr' else out

    def release(self):
        if self.owns_matrix:
            self.matrix.release()


class KernelRowsHessian:
    """The Hessian of an SVM dual that is never stored: SMO computes the rows it needs from X on the device (K12,
    ``svmb200_smo_create_rows``).  ``Q_st = s_s s_t k(x_{s mod n}, x_{t mod n})``: ``layout='plain'`` with ``signs`` = the
    labels (SVC), ``layout='svr'`` with the block signs ``e = [1, -1]`` (SVR).  ``spec`` = ``(kernel id, gamma, coef0,
    degree)`` as ``gram_spec`` resolved it.  Holds ``X`` (a :class:`DeviceMatrix`) until :meth:`release`, and the host copy
    of X that :meth:`product` evaluates against; ``cache_bytes`` sizes the solver's row cache."""

    def __init__(self, ctx, X_device, X_host, spec, layout='plain', signs=None, cache_bytes=0):
        self.ctx, self.X, self.layout = ctx, X_device, layout
        self.X_host = np.ascontiguousarray(X_host, dtype=np.float64)
        self.n = X_device.rows
        self.kernel, self.gamma, self.coef0, self.degree = spec
        self.signs = None if signs is None else np.ascontiguousarray(signs, dtype=np.float64).ravel()
        self.cache_bytes = int(cache_bytes)
        self.row0, self.nrows = 0, self.n

    @property
    def nvars(self):
        return 2 * self.n if self.layout == 'svr' else self.n

    @property
    def row_signs(self):
        """the sign row of Q = (s s') o [k(x_s mod n, x_t mod n)]"""
        if self.layout == 'svr':
            return np.hstack((np.ones(self.n), -np.ones(self.n)))
        return np.ones(self.n) if self.signs is None else self.signs

    def shards(self):
        return [self]

    def kernel_rows(self, rows):
        """k(x_r, x_t) for the listed rows r and every t (unsigned), by the device function the solver uses"""
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        ld = N.padded_ld(self.n)
        out = DeviceMatrix(self.ctx, len(rows), self.n, ld)
        try:
            N.call('svmb200_kernel_rows', self.ctx.handle, C.c_void_p(self.X.dptr), self.n, self.X.ld, self.X.cols,
                   int(self.kernel), float(self.gamma), float(self.coef0), float(self.degree),
                   rows.ctypes.data_as(C.c_void_p), len(rows), C.c_void_p(out.dptr), ld)
            return out.to_host()
        finally:
            out.release()

    def to_host(self):
        """The whole Hessian on the host, from svmb200_kernel_rows (small problems: tests)."""
        K = self.kernel_rows(np.arange(self.n))
        if self.layout == 'svr':
            return np.vstack((np.hstack((K, -K)), np.hstack((-K, K))))
        return self.signs[:, None] * K * self.signs[None, :] if self.signs is not None else K

    def product(self, v):
        """Q @ v through K6 (svmb200_decision_device: K1 blocks contracted on the fly), at any n."""
        v = np.asarray(v, dtype=np.float64).ravel()
        s = self.row_signs
        beta = s * v
        beta = beta[:self.n] + beta[self.n:] if self.layout == 'svr' else beta
        out = np.empty(self.n)
        N.call('svmb200_decision_device', self.ctx.handle, C.c_void_p(self.X.dptr), self.n, self.X.ld,
               N.ptr(np.ascontiguousarray(beta)), N.ptr(self.X_host), self.n, self.X.cols, int(self.kernel),
               float(self.gamma), float(self.coef0), float(self.degree), 0.0, N.ptr(out))
        return s * (np.concatenate((out, out)) if self.layout == 'svr' else out)

    def release(self):
        if self.X is not None:
            self.X.release()
            self.X = None


class DeviceGroup:
    """One process, N GPUs: ranks 0..N-1 are contexts of the calling thread (one per device) whose exchange arenas are
    mapped by plain peer access (``svmb200_comm_local_group``).  Problems with at least ``MIN_ROWS_PER_GPU`` rows per GPU
    are row-block sharded over the group exactly like a ``torchrun`` job (same partition, same kernels, same bits);
    smaller ones stay on the solo context -- an exchange per iteration costs more than it saves there."""

    MIN_ROWS_PER_GPU = 512

    def __init__(self, devices, arena_bytes=64 << 20):
        devices = [int(d) for d in devices]
        if len(devices) < 2 or len(set(devices)) != len(devices):
            raise ValueError('a device group needs two or more distinct devices')
        self.ctxs = [Context(device=d) for d in devices]
        handles = (C.c_void_p * len(devices))(*[c.handle.value for c in self.ctxs])
        N.call('svmb200_comm_local_group', handles, len(devices), int(arena_bytes))
        for r, c in enumerate(self.ctxs):
            c.rank, c.nranks = r, len(devices)
        self.devices = devices

    def __len__(self):
        return len(self.ctxs)

    def wants(self, n):
        """shard an n x n matrix over the group?  (every rank must own rows: the fused exchange has no collective)"""
        return _group_shards(len(self.ctxs), n)

    def replicate(self, src):
        """copies of a DeviceMatrix on every rank's device (rank order); the source's own device reuses it in place"""
        out = []
        for c in self.ctxs:
            m = DeviceMatrix(c, src.rows, src.cols, src.ld)
            N.call('svmb200_copy_peer', c.handle, C.c_void_p(m.dptr), src.ctx.handle, C.c_void_p(src.dptr), src.nbytes)
            out.append(m)
        return out

    def sync(self):
        for c in self.ctxs:
            c.sync()

    def trim(self):
        for c in self.ctxs:
            c.trim()


def _group_shards(P, n):
    rows_per_rank = shard_rows(n, 0, P)[1]
    return n >= P * DeviceGroup.MIN_ROWS_PER_GPU and (P - 1) * rows_per_rank < n


class GroupHessian:
    """The n x n matrix of a solve, row-block sharded over the ranks of a :class:`DeviceGroup` (``parts[r]`` is rank r's
    :class:`DeviceHessian`).  Same interface as ``DeviceHessian`` where the solvers and estimators use it."""

    def __init__(self, group, n, layout='plain'):
        self.group, self.n, self.layout = group, int(n), layout
        self.parts = [DeviceHessian(c, n, layout) for c in group.ctxs]
        self.ctx = group.ctxs[0]
        self.ld = self.parts[0].ld
        self.signs = None
        self.row0, self.nrows = 0, self.n

    @property
    def nvars(self):
        return 2 * self.n if self.layout == 'svr' else self.n

    @property
    def matrix(self):
        return self.parts[0].matrix

    def shards(self):
        return self.parts

    def with_signs(self, signs):
        raise NotImplementedError('signed views (lockstep one-vs-rest batches) are not available on a device group')

    @classmethod
    def from_host(cls, group, Q):
        Q = np.asarray(Q, dtype=np.float64)
        n = Q.shape[0]
        H = cls(group, n, 'plain')
        for part in H.parts:
            block = np.zeros((max(part.nrows, 1), part.ld))
            block[:part.nrows, :n] = Q[part.row0:part.row0 + part.nrows]
            part.ctx.h2d(part.matrix.dptr, block)
        return H

    def shard_to_host(self):
        return np.vstack([p.shard_to_host() for p in self.parts])

    def to_host(self):
        M = self.shard_to_host()
        if self.layout == 'svr':
            return np.vstack((np.hstack((M, -M)), np.hstack((-M, M))))
        return M

    def product(self, v):
        """Q @ v: every rank's shard streams concurrently (svmb200_masked_product_group), one host result"""
        v = np.asarray(v, dtype=np.float64).ravel()
        beta = np.ascontiguousarray(v[:self.n] - v[self.n:] if self.layout == 'svr' else v)
        out = np.empty(self.n)
        P = len(self.parts)
        ctxs = (C.c_void_p * P)(*[p.ctx.handle.value for p in self.parts])
        mats = (C.c_void_p * P)(*[p.matrix.dptr for p in self.parts])
        N.call('svmb200_masked_product_group', ctxs, mats, P, self.n, self.ld, N.ptr(beta), N.ptr(out))
        return np.concatenate((out, -out)) if self.layout == 'svr' else out

    def release(self):
        for p in self.parts:
            p.release()


def make_hessian(ctx, n, layout='plain'):
    """The resident matrix of an n-variable problem: sharded over ``ctx.group`` when there is one and the problem is
    large enough, on ``ctx`` (this rank's row shard under torchrun) otherwise."""
    if ctx.group is not None and ctx.group.wants(n):
        return GroupHessian(ctx.group, n, layout)
    return DeviceHessian(ctx, n, layout)


def hessian_from_host(ctx, Q):
    if ctx.group is not None and ctx.group.wants(np.shape(Q)[0]):
        return GroupHessian.from_host(ctx.group, Q)
    return DeviceHessian.from_host(ctx, Q)


_symmetric = None   # None: the library's default (environment variable SVMB200_SYMMETRIC, else off)


def use_symmetric_pass(on=True):
    """Opt in to (or out of) the symmetric pass: solvers that hold their whole Hessian on one GPU take every product
    ``Q d`` from the UPPER TRIANGLE of the matrix alone -- half the HBM bytes per iteration, about twice the iterations
    per second on a bandwidth-bound fit.  Every Hessian of the SVM dual is symmetric, so this is always valid for the
    estimators; for a hand-made ``Quadratic`` the caller vouches for it.  The iterate is reproducible run to run but
    follows another summation order than the default pass, so it is NOT bit-identical to it (well-conditioned problems
    stay far inside the 1e-8 of ``north_star``; the default keeps the bit-exact contract).  ``SVMB200_SYMMETRIC=1`` in
    the environment does the same without a code change."""
    global _symmetric
    _symmetric = bool(on)
    if _default_ctx is not None:
        N.call('svmb200_ctx_set_symmetric', _default_ctx.handle, int(_symmetric))
        if _default_ctx.group is not None:   # one process, N GPUs: the pass is sharded over the group's contexts
            for c in _default_ctx.group.ctxs:
                N.call('svmb200_ctx_set_symmetric', c.handle, int(_symmetric))


_devices = None


def use_devices(devices):
    """Fan large problems of this process out to these GPUs (``None`` / one device: single-GPU).  The environment variable
    ``SVMB200_DEVICES`` (comma-separated indices, or ``all``) does the same without a code change.  Not for ``torchrun``
    jobs: there every rank owns one GPU already."""
    global _devices, _default_ctx
    _devices = None if devices is None else [int(d) for d in devices]
    if _default_ctx is not None and _default_ctx.nranks == 1:
        _attach_group(_default_ctx)


def _configured_devices():
    if _devices is not None:
        return _devices
    env = os.environ.get('SVMB200_DEVICES', '').strip()
    if not env:
        return None
    if env.lower() == 'all':
        count = C.c_int(0)
        N.call('svmb200_device_count', C.byref(count))
        return list(range(count.value))
    return [int(t) for t in env.split(',') if t.strip() != '']


def _attach_group(ctx):
    devs = _configured_devices()
    if devs is None or len(devs) < 2:
        if ctx.group is not None:
            ctx.group = None
        return
    if ctx.group is None or ctx.group.devices != devs:
        ctx.group = DeviceGroup(devs)


def default_context():
    """Process-wide context.  Under ``torchrun`` (torch.distributed initialised, world size > 1) the
    context joins an NCCL communicator whose id is broadcast through torch.distributed."""
    global _default_ctx
    if _default_ctx is not None:
        return _default_ctx
    devs = _configured_devices()
    ctx = Context(device=devs[0]) if devs else Context()
    distributed = False
    import sys
    if 'torch' in sys.modules:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            rank, world = dist.get_rank(), dist.get_world_size()
            distributed = True
            ctx.attach_communicator(rank, world, broadcast_unique_id(dist, Context.new_unique_id))
            if os.environ.get('SVMB200_EXCHANGE', 'p2p').lower() != 'nccl':
                ctx.enable_peer_exchange(dist)
    if not distributed:
        _attach_group(ctx)
    _default_ctx = ctx
    return ctx


def would_shard(n):
    """Would the Hessian of an n-variable fit started now be row-sharded (torchrun world > 1, or a device group that
    shards n)?  Answered without creating a context."""
    if _default_ctx is not None:
        return _default_ctx.nranks > 1 or (_default_ctx.group is not None and _default_ctx.group.wants(int(n)))
    import sys
    if 'torch' in sys.modules:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return True
    devs = _configured_devices()
    return devs is not None and len(devs) >= 2 and _group_shards(len(devs), int(n))


def broadcast_unique_id(dist, make_id):
    """Rank 0 creates the 128-byte NCCL id, every rank receives it through torch.distributed."""
    box = [make_id() if dist.get_rank() == 0 else None]
    dist.broadcast_object_list(box, src=0)
    uid = bytes(box[0])
    if len(uid) != 128:
        raise ValueError('NCCL unique id must be 128 bytes')
    return uid


def set_default_context(ctx):
    global _default_ctx
    _default_ctx = ctx
