"""SMO (optimizer='smo') with and without libsvm's shrinking on the same seeded inputs: fits alternated
(shrinking=False, shrinking=True, ...), --reps fits per arm after one warm-up fit of each, medians.  One JSON line per
workload: iterations, us per iteration, solve and fit time, the active share at the last shrink check, shrink checks,
gradient reconstructions, and the relative difference of the two dual objectives (FP64, the fits' own f_x), with the
GPU's name and power limit read in the same call.
    python scripts/bench_smo_shrinking.py [--workloads C1,C4,C4-computed,C2,C5-200k,C4-search] [--reps 3] [--tol 1e-3]
C4-search is a grid search of 5 folds x 6 values of C at C4 (K14 batches the fold problems), timed end to end.
The time of the reconstructions is not separated from the solve: they run inside the cooperative kernel."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))

from bench_smo import gpu_info  # noqa: E402

WORKLOADS = {   # name: (config, n, row source)
    'C1': ('C1', None, 'auto'),
    'C4': ('C4', None, 'resident'),
    'C4-computed': ('C4', None, 'computed'),
    'C2': ('C2', None, 'auto'),
    'C5-200k': ('C5', 200_000, 'auto'),
}


def estimator(spec, tol, shrinking, **kw):
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import hinge, epsilon_insensitive
    if spec['task'] == 'svc':
        return SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=10 ** 7,
                   shrinking=shrinking, **kw)
    return SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=spec['degree']), C=1, epsilon=spec['epsilon'],
               dual=True, optimizer='smo', tol=tol, max_iter=10 ** 7, shrinking=shrinking, **kw)


def one_fit(spec, X, y, tol, shrinking):
    from optiml_b200.runtime import default_context
    ctx = default_context()
    m = estimator(spec, tol, shrinking)
    ctx.sync()
    t0 = time.perf_counter()
    m.fit(X, y)
    ctx.sync()
    wall = time.perf_counter() - t0
    o = m.optimizer
    out = dict(iters=o.iter, status=o.status, solve_ms=o.device_ms, fit_s=wall, f=o.f_x, active=o.active_,
               nvars=len(o.x), checks=o.shrink_checks, reconstructions=o.reconstructions, row_source=o.row_source)
    m.obj.release()
    return out


def fits(name, tol, reps):
    from optiml_b200.configs import make_config
    cfg, n, rows = WORKLOADS[name]
    if rows == 'auto':
        os.environ.pop('SVMB200_SMO_ROWS', None)
    else:
        os.environ['SVMB200_SMO_ROWS'] = rows
    spec, X, y = make_config(cfg, n=n)
    large = len(y) > 100_000
    if not large:   # warm-up: the module, the buffer pools and the kernels' shared-memory settings
        one_fit(spec, X, y, tol, False)
        one_fit(spec, X, y, tol, True)
    runs = {False: [], True: []}
    for _ in range(reps):
        for shrinking in (False, True):
            runs[shrinking].append(one_fit(spec, X, y, tol, shrinking))
    os.environ.pop('SVMB200_SMO_ROWS', None)
    gpu, power = gpu_info()
    row = dict(workload=name, config=cfg, task=spec['task'], n=len(y), tol=tol, reps=reps, gpu=gpu, power_limit=power)
    for shrinking, rs in runs.items():
        key = 'shrinking' if shrinking else 'plain'
        med = lambda k: float(np.median([r[k] for r in rs]))   # noqa: E731
        r0 = rs[0]
        assert all(r['iters'] == r0['iters'] and r['f'] == r0['f'] for r in rs), 'fits of one arm differ'
        row[key] = dict(iters=r0['iters'], status=r0['status'], row_source=r0['row_source'],
                        solve_s=round(med('solve_ms') / 1e3, 4), fit_s=round(med('fit_s'), 4),
                        us_per_iter=round(1e3 * med('solve_ms') / max(r0['iters'], 1), 3),
                        active_share=round(r0['active'] / r0['nvars'], 4), checks=r0['checks'],
                        reconstructions=r0['reconstructions'], f=r0['f'])
    fp, fs = row['plain']['f'], row['shrinking']['f']
    row['f_rel_diff'] = abs(fs - fp) / abs(fp)
    row['fit_speedup'] = round(row['plain']['fit_s'] / row['shrinking']['fit_s'], 3)
    return row


def grid_search(tol, reps):
    from optiml_b200.configs import make_config
    from optiml_b200.model_selection import GridSearchCV
    from optiml_b200.ml.svm import SVC
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.ml.svm.losses import hinge
    spec, X, y = make_config('C4')
    grid = {'C': [0.1, 0.3, 1.0, 3.0, 10.0, 30.0]}

    def run(shrinking):
        est = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=tol, max_iter=10 ** 7,
                  shrinking=shrinking)
        t0 = time.perf_counter()
        s = GridSearchCV(est, grid, cv=5, refit=False).fit(X, y)
        return time.perf_counter() - t0, s.cv_results_['mean_test_score']

    run(False)
    run(True)
    times = {False: [], True: []}
    scores = {}
    for _ in range(reps):
        for shrinking in (False, True):
            t, sc = run(shrinking)
            times[shrinking].append(t)
            scores[shrinking] = sc
    gpu, power = gpu_info()
    tp, ts = float(np.median(times[False])), float(np.median(times[True]))
    return dict(workload='C4-search', config='C4', folds=5, values_of_C=6, tol=tol, reps=reps, gpu=gpu,
                power_limit=power, plain=dict(search_s=round(tp, 3)), shrinking=dict(search_s=round(ts, 3)),
                search_speedup=round(tp / ts, 3),
                max_score_diff=float(np.max(np.abs(scores[False] - scores[True]))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='C1,C4,C4-computed,C2,C5-200k,C4-search')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--tol', type=float, default=1e-3)
    ap.add_argument('--out', default=None, help='also append the lines to this file')
    args = ap.parse_args()
    for name in args.workloads.split(','):
        name = name.strip()
        row = grid_search(args.tol, args.reps) if name == 'C4-search' else fits(name, args.tol, args.reps)
        line = json.dumps(row)
        print(line, flush=True)
        if args.out:
            with open(args.out, 'a') as fh:
                fh.write(line + '\n')


if __name__ == '__main__':
    main()
