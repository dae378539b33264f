"""Device timing of SMO fits that share one Gram matrix (csrc/k_smo.cuh K14, svmb200_smo_run_batch) against sklearn's
clone-per-class fit of the same estimator on the same inputs.

Arms:  `batch`   optiml_b200.ml.multiclass.OneVsRestClassifier / MultiOutputRegressor -- one M in HBM, the problems
                 side by side on disjoint ranges of SMs;
       `cloned`  sklearn.multiclass.OneVsRestClassifier / sklearn.multioutput.MultiOutputRegressor -- one Gram build
                 and one SMO solve per class, one after the other (the reference's recipe, on the GPU).
Workloads:  c4   C4's inputs (n = 50 000, d = 128) in 4 quantile classes of a random projection (scripts/bench_ovr.py),
                 SVC Gaussian, tol 1e-3 -- few problems, each large enough for many CTAs;
            c1   C1-sized inputs (n = 2 000, d = 20) in 10 classes, SVC Gaussian, tol 1e-3 -- many problems, each of
                 which runs best on 16 CTAs or fewer alone;
            svr  C2-shaped inputs (n = 10 000, d = 32, 20 000 variables), 3 targets, SVR cubic polynomial, tol 1e-3.
The arms alternate, `--reps` fits each after one warm-up fit of each.  One JSON line per fit: fit s (wall clock, the
results on the host), solve s (batch: the shared solve; cloned: the sum of the solves), summed problem-iterations,
problem-iterations per solve second, iterations per class; then one line per workload with the medians and whether the
two arms agree bitwise (alpha, G, iterations, status, f history).  `--chunks` sweeps SVMB200_SMO_BATCH_CHUNK in the batch
arm.  The card's name and power limit are read in the same run.

    python scripts/bench_smo_batch.py [--workloads c4,c1,svr] [--reps 3] [--chunks 1024,4096,16384] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in q.split(','))
    return name, power


def workload(name):
    from optiml_b200.configs import make_config
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import epsilon_insensitive, hinge

    def classes(X, k):
        score = X @ np.random.default_rng(0).standard_normal(X.shape[1])
        return np.searchsorted(np.quantile(score, np.linspace(0, 1, k + 1)[1:-1]), score)

    svc = SVC(loss=hinge, kernel=GaussianKernel(), C=1, dual=True, optimizer='smo', tol=1e-3, max_iter=10 ** 7)
    if name == 'c4':
        spec, X, _ = make_config('C4')
        return 'ovr', svc, X, classes(X, 4)
    if name == 'c1':
        spec, X, _ = make_config('C1', n=2000)
        return 'ovr', svc, X, classes(X, 10)
    spec, X, y = make_config('C2')
    est = SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo',
              tol=1e-3, max_iter=10 ** 7)
    return 'mor', est, X, np.stack([y, np.roll(y, 11), 0.5 * y + 1.0], axis=1)


def fit(kind, arm, est, X, Y):
    from sklearn.multiclass import OneVsRestClassifier as SkOVR
    from sklearn.multioutput import MultiOutputRegressor as SkMOR
    from optiml_b200.ml.multiclass import MultiOutputRegressor, OneVsRestClassifier
    cls = {('ovr', 'batch'): OneVsRestClassifier, ('ovr', 'cloned'): SkOVR,
           ('mor', 'batch'): MultiOutputRegressor, ('mor', 'cloned'): SkMOR}[(kind, arm)]
    t0 = time.perf_counter()
    model = cls(est).fit(X, Y)
    fit_s = time.perf_counter() - t0
    ests = model.estimators_
    if arm == 'batch':
        assert all(e.fit_times_.get('batch') == len(ests) for e in ests), 'the batch arm did not run as one batch'
        solve_s = ests[0].fit_times_['solve_s']
    else:
        solve_s = sum(e.fit_times_['solve_s'] for e in ests)
    out = [(e.optimizer.x, e.optimizer.g_x, e.optimizer.iter, e.optimizer.status, e.optimizer.f_hist) for e in ests]
    for e in ests:
        e.obj.release()
    return fit_s, solve_s, out


def same(a, b):
    return all(np.array_equal(u, v) if isinstance(u, np.ndarray) else u == v
               for x, y in zip(a, b) for u, v in zip(x, y))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='c4,c1,svr')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--chunks', default='', help='comma-separated SVMB200_SMO_BATCH_CHUNK values for the batch arm')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    warnings.simplefilter('ignore')
    gpu, power = card()
    sink = open(args.out, 'a') if args.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if sink:
            sink.write(line + '\n')
            sink.flush()

    chunks = [int(c) for c in args.chunks.split(',') if c] or [None]
    for wname in args.workloads.split(','):
        kind, est, X, Y = workload(wname)
        for arm in ('batch', 'cloned'):
            fit(kind, arm, est, X, Y)   # warm-up: module loads, buffer pools
        arms = [('batch', c) for c in chunks] + [('cloned', None)]
        results = {a: [] for a in arms}
        for rep in range(args.reps):
            for arm, chunk in arms:
                if chunk is None:
                    os.environ.pop('SVMB200_SMO_BATCH_CHUNK', None)
                else:
                    os.environ['SVMB200_SMO_BATCH_CHUNK'] = str(chunk)
                fit_s, solve_s, out = fit(kind, arm, est, X, Y)
                iters = [int(o[2]) for o in out]
                results[(arm, chunk)].append((fit_s, solve_s, out))
                emit(dict(workload=wname, arm=arm, chunk=chunk if arm == 'batch' else None, rep=rep, fit_s=round(fit_s, 4),
                          solve_s=round(solve_s, 4), problem_iterations=sum(iters),
                          problem_its_per_s=round(sum(iters) / solve_s, 1), iterations=iters,
                          status=[o[3] for o in out], gpu=gpu, power_limit=power))
        os.environ.pop('SVMB200_SMO_BATCH_CHUNK', None)
        ref = results[('cloned', None)][0][2]
        for (arm, chunk), rs in results.items():
            fs, ss = np.median([r[0] for r in rs]), np.median([r[1] for r in rs])
            its = sum(int(o[2]) for o in rs[0][2])
            emit(dict(workload=wname, summary=True, arm=arm, chunk=chunk, n=int(X.shape[0]), problems=len(ref),
                      median_fit_s=round(float(fs), 4), median_solve_s=round(float(ss), 4), problem_iterations=its,
                      problem_its_per_s=round(its / float(ss), 1),
                      bitwise_equal_to_cloned=all(same(r[2], ref) for r in rs), gpu=gpu, power_limit=power))
    if sink:
        sink.close()


if __name__ == '__main__':
    main()
