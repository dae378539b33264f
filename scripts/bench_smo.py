"""SMO (K11, optimizer='smo') on BASELINE configs C1, C4 (SVC, Gaussian) and C2 (SVR, poly) at full size, one JSON line
per config: iterations, status, final gap, fit time (device events and wall clock), solve time and us per iteration,
matrix bytes per iteration, the GPU's name and power limit -- and a host arm, sklearn.svm.SVC / SVR (libsvm) on the
same kernel, gamma, C and tol, with both dual objectives evaluated in FP64 on the same resident Q.
    python scripts/bench_smo.py [--configs C1,C4,C2] [--tol 1e-3] [--no-sklearn] [--grid G] [--n N]
                                [--rows auto|resident|computed] [--cache-mb MB] [--large]
--grid sets SVMB200_SMO_GRID (CTAs of the cooperative launch; default one per SM) for grid-size sweeps.  --rows and
--cache-mb set SVMB200_SMO_ROWS / SVMB200_SMO_CACHE_MB (the row source, K12, and its row cache; default: the automatic
choice); every line reports the row source, the cache's slots and hit rate and the X bytes one computed row reads.
--large is for sizes only the computed form runs: one fit, no warm-up fit, no sklearn arm."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [t.strip() for t in out.split(',')]
        return name, power
    except (OSError, ValueError, subprocess.SubprocessError):
        return 'unknown', 'unknown'


def dual_objective(H, q, alpha):
    """a'Qa/2 + q'a through one masked product over the resident matrix"""
    return float(0.5 * alpha @ H.product(alpha) + q @ alpha)


def run(name, tol, max_iter, sklearn_arm, n=None, large=False):
    from optiml_b200.configs import make_config
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    from optiml_b200.runtime import default_context
    from oracle.svm_oracle import resolve_gamma
    spec, X, y = make_config(name, n=n)
    n = len(y)
    ctx = default_context()
    for rep in range(1 if large else 2):   # the first fit warms the module, the buffer pools and the kernel's shared-memory setting
        if spec['task'] == 'svc':
            m = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=max_iter)
        else:
            m = SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=spec['degree']), C=1, epsilon=spec['epsilon'],
                    dual=True, optimizer='smo', tol=tol, max_iter=max_iter)
        ctx.sync()
        ctx.timer_start()
        t0 = time.perf_counter()
        m.fit(X, y)
        fit_wall = time.perf_counter() - t0
        fit_dev_ms = ctx.timer_stop_ms()
        if rep == 0:
            m.obj.release()
    o = m.optimizer
    gpu, power = gpu_info()
    row = dict(config=name, task=spec['task'], kernel=spec['kernel'], n=n, nvars=len(o.x), tol=tol,
               grid=os.environ.get('SVMB200_SMO_GRID', 'one CTA per SM'), iters=o.iter, status=o.status, gap=o.gap,
               fit_s_wall=round(fit_wall, 4), fit_ms_device=round(fit_dev_ms, 2), solve_ms_device=round(o.device_ms, 2),
               us_per_iter=round(1e3 * o.device_ms / max(o.iter, 1), 3), matrix_bytes_per_iter=16 * n,
               n_sv=int(len(m.support_)), f=o.f_x, gpu=gpu, power_limit=power, row_source=o.row_source,
               cache_slots=o.cache_slots, cache_hits=o.cache_hits, cache_misses=o.cache_misses,
               hit_rate=round(o.cache_hits / max(o.cache_hits + o.cache_misses, 1), 5),
               x_bytes_per_miss=n * X.shape[1] * 8)
    if sklearn_arm:
        from sklearn.svm import SVC as SkSVC, SVR as SkSVR
        gamma = resolve_gamma('scale', X)
        kw = dict(C=1, tol=tol, gamma=gamma, cache_size=8000)
        if spec['task'] == 'svc':
            sk = SkSVC(kernel='rbf', **kw)
        else:
            sk = SkSVR(kernel='poly', degree=spec['degree'], coef0=0., epsilon=spec['epsilon'], **kw)
        t0 = time.perf_counter()
        sk.fit(X, y)
        sk_wall = time.perf_counter() - t0
        coef = np.zeros(n)
        coef[sk.support_] = sk.dual_coef_.ravel()
        a_sk = np.abs(coef) if spec['task'] == 'svc' else np.hstack((np.maximum(coef, 0.), np.maximum(-coef, 0.)))
        H = m.obj.device_hessian()
        f_ours, f_sk = dual_objective(H, o.f.q, o.x), dual_objective(H, o.f.q, a_sk)
        row.update(sklearn_fit_s_wall=round(sk_wall, 3), sklearn_n_iter=int(np.ravel(sk.n_iter_)[0]),
                   host_cores=os.cpu_count(), f_ours_fp64=f_ours, f_sklearn_fp64=f_sk,
                   f_rel_diff=abs(f_ours - f_sk) / abs(f_sk), intercept=float(m.intercept_),
                   sklearn_intercept=float(np.ravel(sk.intercept_)[0]))
    m.obj.release()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='C1,C4,C2')
    ap.add_argument('--tol', type=float, default=1e-3)
    ap.add_argument('--max-iter', type=int, default=10 ** 7)
    ap.add_argument('--no-sklearn', action='store_true', help='skip the host arm (long configs)')
    ap.add_argument('--n', type=int, default=None, help='sample count (default: the config\'s full size)')
    ap.add_argument('--grid', type=int, default=None, help='CTAs of the cooperative launch (SVMB200_SMO_GRID)')
    ap.add_argument('--rows', choices=['auto', 'resident', 'computed'], default='auto', help='row source (K12)')
    ap.add_argument('--cache-mb', type=float, default=None, help='row cache of the computed form (SVMB200_SMO_CACHE_MB)')
    ap.add_argument('--large', action='store_true', help='one fit, no sklearn arm (sizes beyond HBM)')
    args = ap.parse_args()
    if args.rows != 'auto':
        os.environ['SVMB200_SMO_ROWS'] = args.rows
    if args.cache_mb is not None:
        os.environ['SVMB200_SMO_CACHE_MB'] = repr(args.cache_mb)
    if args.grid is not None:
        os.environ['SVMB200_SMO_GRID'] = str(args.grid)
    for name in args.configs.split(','):
        print(json.dumps(run(name.strip(), args.tol, args.max_iter, not (args.no_sklearn or args.large), args.n,
                             args.large)), flush=True)


if __name__ == '__main__':
    main()
