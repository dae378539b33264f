"""Cross-validation folds as masked problems on one shared M (svmb200_smo_create_subset, fit_shared_gram with training
rows, optiml_b200/model_selection.py) on the B200: the sub-Gram identity, folds against their own fits, and grid
searches against sklearn's on iris, C1-sized inputs, a C2-shaped SVR grid and C4's inputs (5 folds x 6 values of C,
every fold against the KKT conditions)."""
import numpy as np
import pytest
from sklearn.datasets import load_iris
from sklearn.model_selection import StratifiedKFold

import smo_batch_checks as SB
import smo_cv_checks as CV
from optiml_b200.configs import make_config

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('kind', ['linear', 'poly', 'gaussian', 'laplacian', 'sigmoid'])
def test_sub_gram_is_the_gram_of_the_rows(kind):
    spec, X, y = make_config('C1', n=3000)
    CV.check_sub_gram(CV.kernels()[kind], X, CV.ragged_rows(len(X), 2), 'svr' if kind == 'poly' else 'plain')


def test_svc_folds_equal_their_own_fits():
    spec, X, y = make_config('C1', n=6000)
    est = SB.svc(CV.kernels()['gaussian'], tol=1e-3, max_iter=10 ** 6)
    ours, _ = CV.check_folds_equal_own_fits(est, X, y, CV.ragged_rows(len(X), 4), params=[{'C': 0.5}, {'C': 2.0}])
    assert CV.shared(ours)


def test_iris_grid_search():
    X, y = load_iris(return_X_y=True)
    X, y = X[y > 0], y[y > 0]
    ours, _ = CV.grid_search_both(SB.svc(tol=1e-3), {'C': [0.1, 0.3, 1.0, 3.0, 10.0, 30.0]}, X, y, cv=5,
                                  return_train_score=True)
    assert ours.best_score_ >= 0.9


def test_c1_grid_search():
    spec, X, _ = make_config('C1')
    y = (SB.quantile_classes(X, 10) == 0).astype(int)   # one class of ten against the rest
    CV.grid_search_both(SB.svc(tol=1e-3, max_iter=10 ** 6), {'C': [0.1, 0.3, 1.0, 3.0, 10.0, 30.0]}, X, y, cv=5,
                        scoring=['accuracy', 'balanced_accuracy'], refit='balanced_accuracy')


def test_c2_svr_epsilon_by_c_grid():
    spec, X, y = make_config('C2', n=4000)
    CV.grid_search_both(SB.svr(tol=1e-3, max_iter=10 ** 6), {'epsilon': [0.05, 0.1, 0.2], 'C': [0.5, 2.0]}, X, y,
                        cv=3)
    CV.cross_validate_both(SB.svr(tol=1e-3, max_iter=10 ** 6), X, y, cv=4, return_train_score=True)


def test_c4_five_folds_by_six_values_of_c():
    from sklearn.metrics import check_scoring
    from optiml_b200.ml.svm.kernels import GaussianKernel
    from optiml_b200.model_selection import _fit_and_score_shared
    tol = 1e-3
    spec, X, y = make_config('C4')
    est = SB.svc(GaussianKernel(1.0 / X.shape[1]), tol=tol, max_iter=10 ** 7)
    grid = {'C': [0.1, 0.2, 0.5, 1.0, 2.0, 5.0]}
    CV.grid_search_both(est, grid, X, y, cv=5, refit=False)
    splits = list(StratifiedKFold(5).split(X, y))
    out = _fit_and_score_shared(est, X, y, [{'C': c} for c in grid['C']], splits, check_scoring(est), False, np.nan,
                                return_estimator=True)
    fits = [o['estimator'] for o in out]
    assert all(e.fit_times_['batch'] == 30 for e in fits)
    for e, (train, _) in zip(fits, [s for _ in grid['C'] for s in splits]):
        assert e.optimizer.status == 'optimal'
        CV.check_kkt(e, X, y, train, tol)
