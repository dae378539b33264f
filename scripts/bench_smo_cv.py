"""Wall clock of grid searches whose SMO fits share Gram matrices (optiml_b200/model_selection.py) against sklearn's
GridSearchCV over the same estimator on the same inputs.

Arms:  `shared`  optiml_b200.model_selection.GridSearchCV -- one M per kernel spec, built on the union of the training
                 folds; every (candidate, fold) problem a masked problem on it (svmb200_smo_create_subset), all of them
                 side by side in one SMO batch;
       `sklearn` sklearn.model_selection.GridSearchCV -- one clone per (candidate, fold), fitted one after the other:
                 an upload of the fold, a Gram build and one SMO solve each.
Workloads (refit=False: the timed window holds the cross-validation fits alone):
            c4    C4's inputs (n = 50 000, d = 128, binary), SVC Gaussian gamma 1/d, tol 1e-3, 5 folds x 6 values of C;
            c1    C1-sized inputs (n = 2 000, d = 20) in 10 quantile classes of a random projection, class 0 against
                  the rest, SVC Gaussian gamma 'scale' (one M per fold), tol 1e-3, 5 folds x 6 values of C;
            svr   C2-shaped inputs (n = 10 000, d = 32), SVR cubic polynomial, tol 1e-3, 3 folds x 3 epsilon x 2 C;
            iris  iris, versicolor against virginica, SVC Gaussian gamma 'scale', tol 1e-3, 5 folds x 6 values of C.
The arms alternate, `--reps` searches each after one warm-up search of each.  One JSON line per search: wall s, fits,
fits/s, summed problem-iterations and problem-iterations/s (over the wall clock); then one line per workload with the
medians and whether the two arms agree bitwise: cv_results_ without its *_time keys, and every fit's alpha, G,
iteration count and status.  The card's name and power limit are read in the same run.

    python scripts/bench_smo_cv.py [--workloads c4,c1,svr,iris] [--reps 3] [--out FILE]
"""
import argparse
import hashlib
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
    from sklearn.datasets import load_iris
    from optiml_b200.configs import make_config
    from optiml_b200.ml.svm import SVC, SVR
    from optiml_b200.ml.svm.kernels import GaussianKernel, PolyKernel
    from optiml_b200.ml.svm.losses import epsilon_insensitive, hinge

    def svc(gamma):
        return SVC(loss=hinge, kernel=GaussianKernel(gamma), C=1, dual=True, optimizer='smo', tol=1e-3,
                   max_iter=10 ** 7)

    cs = {'C': [0.1, 0.2, 0.5, 1.0, 2.0, 5.0]}
    if name == 'c4':
        spec, X, y = make_config('C4')
        return svc(1.0 / X.shape[1]), cs, X, y, 5
    if name == 'c1':
        spec, X, _ = make_config('C1', n=2000)
        score = X @ np.random.default_rng(0).standard_normal(X.shape[1])
        classes = np.searchsorted(np.quantile(score, np.linspace(0, 1, 11)[1:-1]), score)
        return svc('scale'), cs, X, (classes == 0).astype(int), 5
    if name == 'iris':
        X, y = load_iris(return_X_y=True)
        return svc('scale'), cs, X[y > 0], y[y > 0], 5
    spec, X, y = make_config('C2')
    est = SVR(loss=epsilon_insensitive, kernel=PolyKernel(degree=3), C=1, epsilon=0.1, dual=True, optimizer='smo',
              tol=1e-3, max_iter=10 ** 7)
    return est, {'epsilon': [0.05, 0.1, 0.2], 'C': [0.5, 2.0]}, X, y, 3


class Recorder:
    """every fit's iterations, status and a digest of its alpha and G, taken where both arms finish a fit"""

    def __init__(self):
        from optiml_b200.ml.svm import SVC, SVR
        self.fits, self.saved = [], []
        for cls in (SVC, SVR):
            orig = cls._finish_fit

            def finish(est, plan, _orig=orig):
                out = _orig(est, plan)
                o = est.optimizer
                digest = hashlib.sha256(o.x.tobytes() + o.g_x.tobytes()).hexdigest()
                self.fits.append((int(o.iter), o.status, digest))
                est.obj.release()   # the clone's matrix (shared: one view of M, released with the last clone)
                return out
            self.saved.append((cls, orig))
            cls._finish_fit = finish

    def take(self):
        fits, self.fits = self.fits, []
        return fits


def search(arm, est, grid, X, y, folds, rec):
    from sklearn.model_selection import GridSearchCV as SkGrid
    from optiml_b200.model_selection import GridSearchCV
    cls = GridSearchCV if arm == 'shared' else SkGrid
    t0 = time.perf_counter()
    model = cls(est, grid, cv=folds, refit=False).fit(X, y)
    wall = time.perf_counter() - t0
    results = {k: v for k, v in model.cv_results_.items() if not k.endswith('_time')}
    return wall, results, rec.take()


def same_results(a, b):
    if list(a) != list(b):
        return False
    for k in a:
        u, v = a[k], b[k]
        if isinstance(u, np.ma.MaskedArray):
            if not np.array_equal(np.ma.getmaskarray(u), np.ma.getmaskarray(v)):
                return False
            u, v = np.ma.getdata(u), np.ma.getdata(v)
        if isinstance(u, np.ndarray) and u.dtype.kind == 'f':
            if u.dtype != v.dtype or not np.array_equal(u, v, equal_nan=True):
                return False
        elif len(u) != len(v) or not all(p == q for p, q in zip(u, v)):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='c4,c1,svr,iris')
    ap.add_argument('--reps', type=int, default=3)
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

    rec = Recorder()
    for wname in args.workloads.split(','):
        est, grid, X, y, folds = workload(wname)
        for arm in ('shared', 'sklearn'):
            search(arm, est, grid, X, y, folds, rec)   # warm-up: module loads, buffer pools
        runs = {'shared': [], 'sklearn': []}
        for rep in range(args.reps):
            for arm in ('shared', 'sklearn'):
                wall, results, fits = search(arm, est, grid, X, y, folds, rec)
                runs[arm].append((wall, results, fits))
                its = sum(f[0] for f in fits)
                emit(dict(workload=wname, arm=arm, rep=rep, wall_s=round(wall, 4), fits=len(fits),
                          fits_per_s=round(len(fits) / wall, 3), problem_iterations=its,
                          problem_its_per_s=round(its / wall, 1), status=sorted({f[1] for f in fits}), gpu=gpu,
                          power_limit=power))
        ref_results, ref_fits = runs['sklearn'][0][1], sorted(runs['sklearn'][0][2])
        for arm, rs in runs.items():
            wall = float(np.median([r[0] for r in rs]))
            fits = rs[0][2]
            its = sum(f[0] for f in fits)
            emit(dict(workload=wname, summary=True, arm=arm, n=int(X.shape[0]), fits=len(fits), folds=folds,
                      median_wall_s=round(wall, 4), fits_per_s=round(len(fits) / wall, 3), problem_iterations=its,
                      problem_its_per_s=round(its / wall, 1),
                      bitwise_equal_to_sklearn=all(same_results(r[1], ref_results) and sorted(r[2]) == ref_fits
                                                   for r in rs),
                      gpu=gpu, power_limit=power))
        s, k = (float(np.median([r[0] for r in runs[a]])) for a in ('shared', 'sklearn'))
        emit(dict(workload=wname, speedup=round(k / s, 3), gpu=gpu, power_limit=power))
    if sink:
        sink.close()


if __name__ == '__main__':
    main()
