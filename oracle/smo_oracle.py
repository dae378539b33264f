"""NumPy restatement of the SMO solver of csrc/k_smo.cuh  --  TEST INFRASTRUCTURE ONLY (nothing under optiml_b200/ imports it).

libsvm's solver without shrinking (Fan, Chen & Lin 2005, working-set selection WSS2) for

    min a'Qa/2 + q'a   s.t.  y'a = 0,  0 <= a <= C

written for clarity: O(nvars) vector operations per iteration.  Every scalar and vector operation is performed in the
order the kernel performs it, with one IEEE rounding per operation (NumPy does not contract a*b + c), so a run on the
matrix the kernel read replays the device trajectory bit for bit: alpha, G, iteration count, status, both histories.
"""
from dataclasses import dataclass

import numpy as np

TAU = 1e-12


@dataclass
class SMOResult:
    x: np.ndarray          # alpha
    g: np.ndarray          # G = Q alpha + q
    f_hist: np.ndarray     # objective at every evaluated state 0 .. iter
    gap_hist: np.ndarray   # m - M at every evaluated state
    iter: int
    status: str            # 'optimal' or 'stopped'
    rho: float
    f_x: float             # 1/2 sum alpha_t (G_t + q_t)


def full_q(M, layout='plain'):
    """The solver's Hessian from the resident matrix: M itself (plain), or [[M, -M], [-M, M]] (svr)."""
    M = np.asarray(M, dtype=np.float64)
    if layout == 'svr':
        return np.block([[M, -M], [-M, M]])
    return M


def calculate_rho(alpha, G, y, C):
    """libsvm's Solver::calculate_rho: mean of y_t G_t over the free variables, else the middle of [lb, ub]."""
    yG = y * G
    free = (alpha > 0) & (alpha < C)
    if np.any(free):
        return float(np.sum(yG[free]) / np.count_nonzero(free))
    at_lo, at_hi = alpha <= 0, alpha >= C
    ub_set = ((y > 0) & at_lo) | ((y < 0) & at_hi)
    lb_set = ((y > 0) & at_hi) | ((y < 0) & at_lo)
    ub = np.min(yG[ub_set]) if np.any(ub_set) else np.inf
    lb = np.max(yG[lb_set]) if np.any(lb_set) else -np.inf
    return float((ub + lb) / 2)


def _last_argmax(v, mask):
    """largest index among the maxima of v over mask (libsvm's >= scan), or -1"""
    idx = np.flatnonzero(mask)
    if idx.size == 0:
        return -1
    vals = v[idx]
    return int(idx[np.flatnonzero(vals == vals.max())[-1]])


def smo(Q, q, y, C, tol=1e-3, max_iter=10 ** 7):
    """Q: the full (nvars x nvars) Hessian as the kernel reads it (row s holds Q[s][t]); q, y (+-1), C: nvars vectors or
    scalars.  Returns an :class:`SMOResult`."""
    Q = np.asarray(Q, dtype=np.float64)
    nv = Q.shape[0]
    q = np.broadcast_to(np.asarray(q, dtype=np.float64), (nv,)).copy()
    y = np.broadcast_to(np.asarray(y, dtype=np.float64), (nv,)).copy()
    C = np.broadcast_to(np.asarray(C, dtype=np.float64), (nv,)).copy()
    QD = np.diagonal(Q).copy()
    alpha = np.zeros(nv)
    G = q.copy()
    f = 0.0
    f_hist, gap_hist = [], []
    k, status = 0, None
    while True:
        # selection of i
        up = np.where(y > 0, alpha < C, alpha > 0)
        minus_yG = -(y * G)
        i = _last_argmax(minus_yG, up)
        m = minus_yG[i] if i >= 0 else -np.inf
        # selection of j, and M
        low = np.where(y > 0, alpha > 0, alpha < C)
        M = (np.min(minus_yG[low]) if np.any(low) else np.inf) + 0.0
        j = -1
        if i >= 0:
            Qi = Q[i]
            b = m + y * G
            a = (QD[i] + QD) - (2.0 * y[i] * y) * Qi
            a = np.where(a <= 0, TAU, a)
            with np.errstate(divide='ignore', invalid='ignore'):
                key = (b * b) / a
            j = _last_argmax(key, low & (b > 0))
        gap = m - M
        f_hist.append(f)
        gap_hist.append(gap)
        if j < 0 or gap < tol:
            status = 'optimal'
            break
        if k >= max_iter:
            status = 'stopped'
            break
        # libsvm's two-variable step on the signed Q
        qij = Q[i, j]
        ai0, aj0, Ci, Cj = alpha[i], alpha[j], C[i], C[j]
        ai, aj = ai0, aj0
        if y[i] != y[j]:
            quad = (QD[i] + QD[j]) + 2.0 * qij
            if quad <= 0:
                quad = TAU
            delta = (-G[i] - G[j]) / quad
            diff = ai - aj
            ai += delta
            aj += delta
            if diff > 0:
                if aj < 0:
                    aj, ai = 0.0, diff
            elif ai < 0:
                ai, aj = 0.0, -diff
            if diff > Ci - Cj:
                if ai > Ci:
                    ai, aj = Ci, Ci - diff
            elif aj > Cj:
                aj, ai = Cj, Cj + diff
        else:
            quad = (QD[i] + QD[j]) - 2.0 * qij
            if quad <= 0:
                quad = TAU
            delta = (G[i] - G[j]) / quad
            s = ai + aj
            ai -= delta
            aj += delta
            if s > Ci:
                if ai > Ci:
                    ai, aj = Ci, s - Ci
            elif aj < 0:
                aj, ai = 0.0, s
            if s > Cj:
                if aj > Cj:
                    aj, ai = Cj, s - Cj
            elif ai < 0:
                ai, aj = 0.0, s
        dai, daj = ai - ai0, aj - aj0
        lin = dai * G[i] + daj * G[j]
        sq = (dai * dai) * QD[i] + (daj * daj) * QD[j]
        f = f + ((lin + 0.5 * sq) + (dai * daj) * qij)
        alpha[i], alpha[j] = ai, aj
        G = G + (Qi * dai + Q[j] * daj)
        k += 1
    return SMOResult(x=alpha, g=G, f_hist=np.array(f_hist), gap_hist=np.array(gap_hist), iter=k, status=status,
                     rho=calculate_rho(alpha, G, y, C), f_x=float(0.5 * np.dot(alpha, G + q)))
