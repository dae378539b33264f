"""NumPy restatement of the SMO solver of csrc/k_smo.cuh WITH SHRINKING  --  TEST INFRASTRUCTURE ONLY.

``smo(..., shrinking=False)`` is oracle/smo_oracle.py's solver, unchanged.  ``shrinking=True`` adds libsvm's
Solver::do_shrinking / be_shrunk / reconstruct_gradient on the project's conventions (ties to the larger index, no index
permutation: the active set is a flag per variable and every scan stays in index order), as k_smo.cuh runs it:

* l = the variables of the problem, P = min(l, 1000); one ``active`` flag per variable (all set), ``unshrunk`` false and
  a counter at P + 1.  Before the selection of every state the counter is decremented; at 0 it is set back to P and
  the state is a shrink check: m = max -y_t G_t over the active I_up, M = min over the active I_low (the values the
  selection would compute); if not ``unshrunk`` and m - M <= 10 tol: set ``unshrunk``, reconstruct, activate all; then
  deactivate each active variable at a bound that is only in I_low with -y_t G_t > m, or only in I_up with -y_t G_t < M.
* WSS2, the step and the G update run over the active variables only (an inactive G is not updated).
* When the stopping test fires with inactive variables: reconstruct, activate all, counter = 1, select again at the same
  state (no step, k stays; the history of state k is the evaluation that decided it); stop only if it fires again.  A
  max_iter stop with inactive variables reconstructs before G is returned.
* Reconstruct: for every inactive t, G_t = q_t, then for j ascending over alpha_j > 0, G_t = G_t + Q_jt alpha_j (Q_jt
  read from row j; one rounding per product and per sum).

Every operation has one IEEE rounding in the kernel's order, so a run on the matrix the kernel read replays the device
trajectory bit for bit.
"""
from dataclasses import dataclass

import numpy as np

from oracle import smo_oracle as SO

SHRINK_EVERY = 1000


@dataclass
class ShrinkResult(SO.SMOResult):
    active: int = 0            # active variables after the last shrink check
    checks: int = 0
    reconstructions: int = 0


def smo(Q, q, y, C, tol=1e-3, max_iter=10 ** 7, shrinking=False):
    """oracle/smo_oracle.py's ``smo``; with ``shrinking=True`` libsvm's shrinking (module docstring), returning a
    :class:`ShrinkResult`."""
    if not shrinking:
        return SO.smo(Q, q, y, C, tol=tol, max_iter=max_iter)
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
    P = min(nv, SHRINK_EVERY)
    active = np.ones(nv, dtype=bool)
    unshrunk, counter = False, P + 1
    n_active, checks, recons = nv, 0, 0

    def reconstruct():
        rebuild = ~active
        if np.any(rebuild):
            g = q[rebuild].copy()
            for j in np.flatnonzero(alpha > 0):
                g = g + Q[j, rebuild] * alpha[j]
            G[rebuild] = g
        active[:] = True

    k, status, reselect = 0, None, False
    while True:
        if not reselect:
            counter -= 1
            if counter == 0:
                counter = P
                checks += 1
                up = np.where(y > 0, alpha < C, alpha > 0)
                low = np.where(y > 0, alpha > 0, alpha < C)
                minus_yG = -(y * G)
                m = np.max(minus_yG[up & active]) if np.any(up & active) else -np.inf
                M = (np.min(minus_yG[low & active]) if np.any(low & active) else np.inf) + 0.0
                if not unshrunk and m - M <= 10.0 * tol:
                    unshrunk = True
                    reconstruct()
                    recons += 1
                    minus_yG = -(y * G)
                shrink = (low & ~up & (minus_yG > m)) | (up & ~low & (minus_yG < M))
                active &= ~shrink
                n_active = int(np.count_nonzero(active))
        reselect = False
        # WSS2 over the active variables (oracle/smo_oracle.py's selection)
        up = np.where(y > 0, alpha < C, alpha > 0) & active
        minus_yG = -(y * G)
        i = SO._last_argmax(minus_yG, up)
        m = minus_yG[i] if i >= 0 else -np.inf
        low = np.where(y > 0, alpha > 0, alpha < C) & active
        M = (np.min(minus_yG[low]) if np.any(low) else np.inf) + 0.0
        j = -1
        if i >= 0:
            Qi = Q[i]
            b = m + y * G
            a = (QD[i] + QD) - (2.0 * y[i] * y) * Qi
            a = np.where(a <= 0, SO.TAU, a)
            with np.errstate(divide='ignore', invalid='ignore'):
                key = (b * b) / a
            j = SO._last_argmax(key, low & (b > 0))
        gap = m - M
        if len(f_hist) == k + 1:   # a second evaluation of state k decides it
            f_hist[k], gap_hist[k] = f, gap
        else:
            f_hist.append(f)
            gap_hist.append(gap)
        if j < 0 or gap < tol:
            if not np.all(active):
                reconstruct()
                recons += 1
                counter, reselect = 1, True
                continue
            status = 'optimal'
            break
        if k >= max_iter:
            if not np.all(active):
                reconstruct()
                recons += 1
            status = 'stopped'
            break
        qij = Q[i, j]
        ai0, aj0, Ci, Cj = alpha[i], alpha[j], C[i], C[j]
        ai, aj = ai0, aj0
        if y[i] != y[j]:
            quad = (QD[i] + QD[j]) + 2.0 * qij
            if quad <= 0:
                quad = SO.TAU
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
                quad = SO.TAU
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
        G[active] = G[active] + (Qi[active] * dai + Q[j][active] * daj)
        k += 1
    return ShrinkResult(x=alpha, g=G, f_hist=np.array(f_hist), gap_hist=np.array(gap_hist), iter=k, status=status,
                        rho=SO.calculate_rho(alpha, G, y, C), f_x=float(0.5 * np.dot(alpha, G + q)), active=n_active,
                        checks=checks, reconstructions=recons)
