"""oracle/smo_oracle.py (the NumPy restatement of csrc/k_smo.cuh) against libsvm through sklearn.svm: the same problem
solved to the same tolerance, on the CPU."""
import pytest

import smo_checks as SC
from oracle import smo_oracle as SO
from optiml_b200.configs import make_config


@pytest.mark.parametrize('task,cfg,n,kind', [('svc', 'C1', 600, 'gaussian'), ('svc', 'C1', 600, 'linear'),
                                             ('svc', 'C1', 600, 'poly'), ('svr', 'C2', 400, 'poly')])
def test_oracle_matches_libsvm(task, cfg, n, kind):
    spec, X, y = make_config(cfg, n=n)
    K, Q, q, signs, C, gamma = SC.problem(task, X, y, kind)
    r = SO.smo(Q, q, signs, C, tol=1e-5, max_iter=10 ** 6)
    assert r.status == 'optimal' and len(r.f_hist) == len(r.gap_hist) == r.iter + 1
    sk = SC.sklearn_fit(task, X, y, kind, gamma, tol=1e-5)
    SC.check_against_libsvm(task, X, K, Q, q, signs, C, r.x, r.rho, r.gap_hist[-1], 1e-5, sk)
    # the objective tracked step by step is the one of the final iterate
    assert abs(r.f_hist[-1] - r.f_x) <= 1e-9 * abs(r.f_x)


def test_oracle_stops_at_max_iter():
    spec, X, y = make_config('C1', n=100)
    K, Q, q, signs, C, gamma = SC.problem('svc', X, y, 'gaussian')
    r = SO.smo(Q, q, signs, C, tol=1e-5, max_iter=7)
    assert r.status == 'stopped' and r.iter == 7 and len(r.f_hist) == 8 and r.gap_hist[-1] >= 1e-5
