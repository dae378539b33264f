"""ctypes binding of the svmb200 C ABI (include/svmb200.h).

The shared library is built in-tree by ``optiml_b200/csrc/build.py`` (nvcc, sm_100a).  There is no
fallback: if the library is missing, or no B200-class GPU is visible, every compute call raises.
"""
import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SVMB200_LIB') or os.path.join(_HERE, '_lib', 'libsvmb200.so')

KERNEL_LINEAR, KERNEL_POLY, KERNEL_GAUSSIAN, KERNEL_SIGMOID, KERNEL_LAPLACIAN = 0, 1, 2, 3, 4
HESSIAN_PLAIN, HESSIAN_SVR = 0, 1
STATUS = {0: 'unknown', 1: 'optimal', 2: 'stopped'}
RULES = {'adagrad': 0, 'sgd': 1, 'rmsprop': 2, 'adadelta': 3, 'adam': 4, 'amsgrad': 5, 'adamax': 6}
MOMENTUM = {'none': 0, 'polyak': 1, 'nesterov': 2}

c_dp = C.POINTER(C.c_double)
c_vp = C.c_void_p
i64 = C.c_int64

# name -> (argtypes); every function returns int unless listed in _NON_STATUS
PROTOTYPES = {
    'svmb200_device_count': [C.POINTER(C.c_int)],
    'svmb200_ctx_create': [C.c_int, C.POINTER(c_vp)],
    'svmb200_ctx_destroy': [c_vp],
    'svmb200_ctx_info': [c_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t),
                         C.POINTER(C.c_size_t)],
    'svmb200_malloc': [c_vp, C.c_size_t, C.POINTER(c_vp)],
    'svmb200_free': [c_vp, c_vp],
    'svmb200_memset': [c_vp, c_vp, C.c_int, C.c_size_t],
    'svmb200_h2d': [c_vp, c_vp, c_vp, C.c_size_t],
    'svmb200_d2h': [c_vp, c_vp, c_vp, C.c_size_t],
    'svmb200_d2d': [c_vp, c_vp, c_vp, C.c_size_t],
    'svmb200_sync': [c_vp],
    'svmb200_host_alloc_pinned': [C.c_size_t, C.POINTER(c_vp)],
    'svmb200_host_free_pinned': [c_vp],
    'svmb200_timer_start': [c_vp],
    'svmb200_timer_stop_ms': [c_vp, C.POINTER(C.c_float)],
    'svmb200_launch_count': [c_vp, C.POINTER(C.c_uint64)],
    'svmb200_comm_unique_id': [c_vp],
    'svmb200_comm_init': [c_vp, c_vp, C.c_int, C.c_int],
    'svmb200_comm_destroy': [c_vp],
    'svmb200_comm_p2p_export': [c_vp, C.c_size_t, c_vp],
    'svmb200_comm_p2p_attach': [c_vp, c_vp, C.c_int],
    'svmb200_comm_p2p_enabled': [c_vp, C.POINTER(C.c_int)],
    'svmb200_comm_p2p_disable': [c_vp],
    'svmb200_shard_rows': [i64, C.c_int, C.c_int, C.POINTER(i64), C.POINTER(i64)],
    'svmb200_gram': [c_vp, c_vp, i64, i64, c_vp, i64, i64, i64, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double,
                     c_vp, c_vp, C.c_double, i64, i64, c_vp, i64],
    'svmb200_matvec': [c_vp, c_vp, i64, i64, c_vp, c_vp],
    'svmb200_pg_create': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, c_vp, C.c_double, i64,
                          C.POINTER(c_vp)],
    'svmb200_fw_create': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, c_vp, C.c_double, i64, C.c_double,
                          C.POINTER(c_vp)],
    'svmb200_al_create': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_double,
                          C.c_int, C.c_int, c_vp, c_vp, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, i64,
                          C.POINTER(c_vp)],
    'svmb200_pg_create_signed': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_double, i64,
                                 C.POINTER(c_vp)],
    'svmb200_fw_create_signed': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_double, i64,
                                 C.c_double, C.POINTER(c_vp)],
    'svmb200_al_create_signed': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_double,
                                 C.c_double, C.c_int, C.c_int, c_vp, c_vp, C.c_double, C.c_double, C.c_double,
                                 C.c_double, C.c_double, i64, C.POINTER(c_vp)],
    'svmb200_smo_create': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, C.c_double, i64, C.POINTER(c_vp)],
    'svmb200_smo_create_signed': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, C.c_double, i64,
                                  C.POINTER(c_vp)],
    'svmb200_smo_create_subset': [c_vp, c_vp, i64, i64, i64, i64, C.c_int, c_vp, c_vp, c_vp, c_vp, C.c_double, i64,
                                  C.POINTER(c_vp)],
    'svmb200_smo_run_batch': [C.POINTER(c_vp), C.c_int, C.POINTER(i64), C.POINTER(C.c_int)],
    'svmb200_smo_create_rows': [c_vp, c_vp, i64, i64, i64, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, c_vp,
                                c_vp, c_vp, C.c_double, i64, C.c_size_t, C.POINTER(c_vp)],
    'svmb200_smo_cache_stats': [c_vp, C.POINTER(C.c_int), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)],
    'svmb200_smo_set_shrinking': [c_vp, C.c_int],
    'svmb200_smo_shrink_stats': [c_vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)],
    'svmb200_kernel_rows': [c_vp, c_vp, i64, i64, i64, C.c_int, C.c_double, C.c_double, C.c_double, c_vp, i64, c_vp, i64],
    'svmb200_pg_run_batch': [C.POINTER(c_vp), C.c_int, C.POINTER(i64), C.POINTER(C.c_int)],
    'svmb200_matvec_multi': [c_vp, c_vp, i64, i64, C.POINTER(c_vp), C.POINTER(c_vp), C.c_int],
    'svmb200_al_multipliers': [c_vp, C.POINTER(C.c_double), c_vp, c_vp],
    'svmb200_pg_run': [c_vp, i64, C.POINTER(i64), C.POINTER(C.c_int)],
    'svmb200_pg_state': [c_vp, c_vp, c_vp, C.POINTER(C.c_double), C.POINTER(C.c_double)],
    'svmb200_pg_scalars': [c_vp, c_vp],
    'svmb200_pg_history': [c_vp, c_vp, c_vp, C.POINTER(i64)],
    'svmb200_pg_stats': [c_vp, C.POINTER(C.c_float), C.POINTER(i64), C.POINTER(C.c_float)],
    'svmb200_pg_set_profile': [c_vp, C.c_int],
    'svmb200_pg_stats_ex': [c_vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)],
    'svmb200_pg_profile_samples': [c_vp, C.POINTER(i64)],
    'svmb200_pg_device_x': [c_vp, C.POINTER(c_vp)],
    'svmb200_pg_is_symmetric': [c_vp, C.POINTER(C.c_int)],
    'svmb200_pg_set_self_gram': [c_vp, C.c_int],
    'svmb200_pg_is_exact_symv': [c_vp, C.POINTER(C.c_int)],
    'svmb200_matvec_exact': [c_vp, c_vp, i64, i64, c_vp, c_vp],
    'svmb200_exact_symv_geometry': [i64, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)],
    'svmb200_symv': [c_vp, c_vp, i64, i64, c_vp, c_vp],
    'svmb200_ctx_set_symmetric': [c_vp, C.c_int],
    'svmb200_ctx_get_symmetric': [c_vp, C.POINTER(C.c_int)],
    'svmb200_symv_geometry': [i64, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)],
    'svmb200_symv_plan_items': [i64, i64, C.c_int, C.c_int, C.c_int, c_vp, i64, C.POINTER(i64), C.POINTER(i64)],
    'svmb200_symv_plan_info': [i64, i64, C.c_int, C.c_int, C.c_int, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64),
                               C.POINTER(C.c_double)],
    'svmb200_pg_destroy': [c_vp],
    'svmb200_copy_peer': [c_vp, c_vp, c_vp, c_vp, C.c_size_t],
    'svmb200_comm_local_group': [C.POINTER(c_vp), C.c_int, C.c_size_t],
    'svmb200_pg_start_group': [C.POINTER(c_vp), C.c_int],
    'svmb200_pg_run_group': [C.POINTER(c_vp), C.c_int, i64, C.POINTER(i64), C.POINTER(C.c_int)],
    'svmb200_masked_product_group': [C.POINTER(c_vp), C.POINTER(c_vp), C.c_int, i64, i64, c_vp, c_vp],
    'svmb200_masked_product': [c_vp, c_vp, i64, i64, i64, i64, c_vp, c_vp],
    'svmb200_decision': [c_vp, c_vp, i64, c_vp, c_vp, i64, i64, C.c_int, C.c_double, C.c_double, C.c_double,
                         C.c_double, c_vp],
    'svmb200_decision_device': [c_vp, c_vp, i64, i64, c_vp, c_vp, i64, i64, C.c_int, C.c_double, C.c_double, C.c_double,
                                C.c_double, c_vp],
    'svmb200_device_variance': [c_vp, c_vp, i64, i64, i64, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int)],
    'svmb200_gather_rows': [c_vp, c_vp, i64, i64, i64, c_vp, i64, c_vp, i64],
    'svmb200_kernel_matrix_host': [c_vp, c_vp, i64, c_vp, i64, i64, C.c_int, C.c_double, C.c_double, C.c_double,
                                   c_vp],
    'svmb200_host_variance': [c_vp, i64, C.c_int, C.POINTER(C.c_double)],
    'svmb200_host_gather_rows': [c_vp, i64, c_vp, i64, c_vp, C.c_int],
    'svmb200_bcqp_pg_host': [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, i64, C.c_double, i64, c_vp, c_vp, c_vp, c_vp,
                             C.POINTER(i64), C.POINTER(C.c_int)],
}
_NON_STATUS = {
    'svmb200_last_error': ([], C.c_char_p),
    'svmb200_version': ([], C.c_char_p),
    'svmb200_padded_ld': ([i64], i64),
    'svmb200_smo_max_vars': ([C.c_int], i64),
}

_lib = None
_lock = threading.RLock()   # re-entrant: see load_library


class NativeError(RuntimeError):
    """Raised when a svmb200 call fails; carries the library's error text."""


def load_library():
    """Load libsvmb200.so (once).  Raises if it has not been built -- there is no CPU path."""
    global _lib
    # Fast path without the lock: finalizers of device objects (runtime._free_quiet) call this from the garbage
    # collector, which can run at ANY allocation -- also while this very function holds the lock on the same thread.
    # With a plain Lock taken on every call that self-deadlocked (seen once in the CPU suite, as a 120 s stall).
    lib = _lib
    if lib is not None:
        return lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeError(f'{LIB_PATH} not found: build it with `python -m optiml_b200.csrc.build` '
                              '(or __graft_entry__.build()); optiml_b200 has no CPU fallback')
        lib = bind_prototypes(C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL))
        version = lib.svmb200_version().decode()
        if 'sm_100a' not in version:
            # e.g. SVMB200_LIB pointing at the host emulation the test-suite builds: not a compute path
            raise NativeError(f'{LIB_PATH} is not the sm_100a build ({version!r}); optiml_b200 has no CPU fallback')
        _lib = lib
        return _lib


def bind_prototypes(lib):
    """Declare the argument / result types of every entry point of include/svmb200.h on a loaded library."""
    for name, argtypes in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    for name, (argtypes, restype) in _NON_STATUS.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    return lib


def exported_symbols():
    return sorted(list(PROTOTYPES) + list(_NON_STATUS))


def check(rc, what=''):
    if rc != 0:
        msg = load_library().svmb200_last_error().decode(errors='replace')
        raise NativeError(f'{what or "svmb200"} failed (code {rc}): {msg}')


def call(name, *args):
    lib = load_library()
    check(getattr(lib, name)(*args), name)


def as_f64(a, copy=False):
    a = np.array(a, dtype=np.float64, order='C', copy=True) if copy else np.ascontiguousarray(a, dtype=np.float64)
    return a


def ptr(a):
    """void* of a C-contiguous float64 ndarray (or None)."""
    if a is None:
        return None
    assert a.flags['C_CONTIGUOUS'] and a.dtype == np.float64
    return a.ctypes.data_as(c_vp)


def padded_ld(ncols):
    return int(load_library().svmb200_padded_ld(int(ncols)))
