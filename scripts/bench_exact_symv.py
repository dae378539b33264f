#!/usr/bin/env python
"""The product w = Q u of the headline fit on one GPU, full pass (K2, svmb200_matvec) against the exact symmetric pass
(K2e, svmb200_matvec_exact), alternated on the same resident C4 Hessian (DualSVC Gaussian, n = 50 000, d = 128, label
signs): CUDA-event time per product, the bytes each pass moves (K2: the whole n x ld matrix; K2e: the blocks it reads plus
the column chains written and read back, from svmb200_exact_symv_geometry) and the rate.  Every product of both passes
must give the same bits.  Prints one JSON line; the GPU name and power limit go with the numbers.

    python scripts/bench_exact_symv.py [--n N] [--rounds R] [--per-round K]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=50000)
    ap.add_argument('--rounds', type=int, default=10)
    ap.add_argument('--per-round', type=int, default=25)
    args = ap.parse_args()
    from optiml_b200 import _native as N
    from optiml_b200.configs import make_config
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.runtime import default_context
    spec, X, y = make_config('C4', n=args.n)
    n, d = X.shape
    ld = N.padded_ld(n)
    ctx = default_context()
    dX = ctx.upload_matrix(X)
    kid, gamma, coef0, degree = GaussianKernel().gram_spec(X)
    dS = ctx.upload_vector(np.where(y > 0, 1.0, -1.0))
    dQ = ctx.malloc(n * ld * 8)
    N.call('svmb200_gram', ctx.handle, C.c_void_p(dX.dptr), n, dX.ld, C.c_void_p(dX.dptr), n, dX.ld, d, 1, kid, gamma, coef0,
           degree, C.c_void_p(dS.dptr), C.c_void_p(dS.dptr), 0.0, 0, n, C.c_void_p(dQ), ld)
    ctx.sync()
    dX.release()
    dS.release()
    rng = np.random.default_rng(0)
    u = np.zeros(ld)
    u[:n] = rng.uniform(-1.0, 1.0, n) * (rng.random(n) < 0.5)   # a projected direction has many zeros
    du, dw = ctx.malloc(8 * ld), [ctx.malloc(8 * n), ctx.malloc(8 * n)]
    ctx.h2d(du, u)
    symbols = ('svmb200_matvec', 'svmb200_matvec_exact')

    def product(which):
        N.call(symbols[which], ctx.handle, C.c_void_p(dQ), n, ld, C.c_void_p(du), C.c_void_p(dw[which]))

    for which in (0, 1):   # warm-up: scratch, tables, module load
        for _ in range(3):
            product(which)
    ctx.sync()
    times = [[], []]
    identical = True
    for _ in range(args.rounds):
        for which in (0, 1):
            ctx.timer_start()
            for _ in range(args.per_round):
                product(which)
            times[which].append(ctx.timer_stop_ms() / args.per_round)
        a, b = np.empty(n), np.empty(n)
        ctx.d2h(a, dw[0])
        ctx.d2h(b, dw[1])
        identical = identical and bool(np.array_equal(a, b))
    mb, sb, items = C.c_int64(), C.c_int64(), C.c_int64()
    N.call('svmb200_exact_symv_geometry', n, ld, C.byref(mb), C.byref(sb), C.byref(items))
    full_bytes = 8 * n * ld
    exact_bytes = mb.value + sb.value

    def leg(ms, nbytes):
        ms = np.array(ms)
        return {'us_per_product': float(np.median(ms) * 1e3), 'us_min': float(ms.min() * 1e3), 'us_max': float(ms.max() * 1e3),
                'bytes': int(nbytes), 'gb_per_s': float(nbytes / (np.median(ms) / 1e3) / 1e9)}

    line = {'what': 'w = Q u on the C4 Hessian, K2 (full pass) vs K2e (exact symmetric pass), alternated',
            'gpu': gpu_info(), 'n': n, 'ld': ld, 'launches_each': args.rounds * args.per_round,
            'timing': 'CUDA events on the library stream around each round of launches; median over rounds',
            'k2': leg(times[0], full_bytes),
            'k2e': dict(leg(times[1], exact_bytes), matrix_bytes=int(mb.value), scratch_bytes=int(sb.value),
                        tile_items=int(items.value)),
            'w_identical': identical}
    line['speedup'] = line['k2']['us_per_product'] / line['k2e']['us_per_product']
    print(json.dumps(line), flush=True)
    ctx.free(du)
    for p in dw:
        ctx.free(p)
    ctx.free(dQ)
    assert identical, 'K2e and K2 products differ'


if __name__ == '__main__':
    main()
