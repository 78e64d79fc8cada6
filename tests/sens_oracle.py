"""Dense FP64 reference for the solution sensitivity (mpc_sensitivity): `solution_sensitivity(U, prob, act_tol)`.

An independent restatement of what csrc/mpc_sens.cuh computes, built only on the oracle's analytic gradient
(`objective_and_sens`, which also gives the node-bound rows d x_k / dU):
  * active set: control bounds and theta / v bounds of nodes 1..N within act_tol (as `kkt_residual`);
  * LICQ from the singular values of the active rows scaled to unit norm;
  * multipliers by least squares on the active rows, stationarity residual and sign tests;
  * the Hessian of the Lagrangian by central differences of its analytic gradient (objective gradient minus the
    multiplier-weighted node rows), d(grad)/dp by central differences in each parameter;
  * SOSC from the eigenvalues of Z^T H Z (Z an orthonormal null-space basis of the active rows);
  * dU from the full KKT matrix by numpy.linalg.solve.
Parameters: p = (vr_b, w_speed, w_control, w_diff); vr_b is the reference speed of the stages k >= vr_n.
"""
from __future__ import annotations

import copy

import numpy as np
import scipy.linalg

from helpers import orc

NOT_STATIONARY, WEAKLY_ACTIVE, DEGENERATE, NOT_SOSC, NONFINITE = 1, 2, 4, 8, 16
NAN_FLAGS = NOT_STATIONARY | DEGENERATE | NOT_SOSC | NONFINITE
LICQ_TOL, SOSC_TOL, WEAK_TOL = 1e-9, 1e-10, 1e-6


def with_param(prob, c, value, vr_n):
    q = copy.copy(prob)
    if c == 0:
        q.ref_v = prob.ref_v.copy()
        q.ref_v[vr_n:] = value
    else:
        setattr(q, ("w_speed", "w_control", "w_input_diff")[c - 1], value)
    return q


def param_values(prob, vr_n):
    vr_b = float(prob.ref_v[vr_n]) if vr_n < prob.N else 0.0
    return [vr_b, prob.w_speed, prob.w_control, prob.w_input_diff]


def active_rows(U, prob, act_tol, S=None, X=None):
    """(rows [m, 2N], descriptors): control rows +-e_i, node rows +-S[k, comp]; + at a lower bound, - at an upper."""
    N = prob.N
    if S is None:
        _, _, X, S = orc.objective_and_sens(U.reshape(-1), prob)
    Uf = U.reshape(-1)
    lim = np.tile([orc.A_MAX, orc.DELTA_MAX], N)
    rows, desc = [], []
    for i in range(2 * N):
        e = np.zeros(2 * N)
        e[i] = 1.0
        if Uf[i] + lim[i] <= act_tol:
            rows.append(e); desc.append(("u", i, 1.0))
        if lim[i] - Uf[i] <= act_tol:
            rows.append(-e); desc.append(("u", i, -1.0))
    for k in range(1, N + 1):
        for comp, (lb, ub) in ((3, (orc.V_MIN, orc.V_MAX)), (2, (orc.TH_MIN, orc.TH_MAX))):
            if X[k, comp] - lb <= act_tol:
                rows.append(S[k, comp].copy()); desc.append(("x", (k, comp), 1.0))
            if ub - X[k, comp] <= act_tol:
                rows.append(-S[k, comp]); desc.append(("x", (k, comp), -1.0))
    return np.array(rows).reshape(-1, 2 * N), desc


def solution_sensitivity(U, prob, act_tol=1e-4, stat_tol=1e-3, vr_n=0, h=1e-5):
    """Returns (jac [2, 4], flags, multipliers [m] in the order of `active_rows`, residual)."""
    N = prob.N
    U = np.asarray(U, np.float64).reshape(N, 2)
    nan_jac = np.full((2, 4), np.nan)
    f, g, X, S = orc.objective_and_sens(U.reshape(-1), prob)
    if not (np.all(np.isfinite(U)) and np.all(np.isfinite(X)) and np.all(np.isfinite(g)) and np.isfinite(f)):
        return nan_jac, NONFINITE, None, np.nan
    A, desc = active_rows(U, prob, act_tol, S, X)
    m = A.shape[0]
    if m:
        norms = np.linalg.norm(A, axis=1)
        if np.any(norms == 0.0) or m > 2 * N:
            return nan_jac, DEGENERATE, None, np.nan
        sv = np.linalg.svd(A / norms[:, None], compute_uv=False)
        if sv.min() <= LICQ_TOL:
            return nan_jac, DEGENERATE, None, np.nan
        mu = np.linalg.lstsq(A.T, g, rcond=None)[0]
    else:
        mu = np.zeros(0)
    res = float(np.linalg.norm(g - A.T @ mu))
    tau = stat_tol * (1 + abs(f))
    flags = NOT_STATIONARY if res > tau else 0
    tw = WEAK_TOL * (1 + abs(f))
    if m and mu.min() < -tw:
        flags |= NOT_STATIONARY
    elif m and mu.min() <= tw:
        flags |= WEAKLY_ACTIVE
    node = [(d[1], d[2], mu[q]) for q, d in enumerate(desc) if d[0] == "x"]

    def grad_l(u, pr):
        _, gg, _, SS = orc.objective_and_sens(u, pr)
        for (k, comp), sg, nu in node:
            gg = gg - nu * sg * SS[k, comp]
        return gg

    u0 = U.reshape(-1)
    H = np.zeros((2 * N, 2 * N))
    for i in range(2 * N):
        e = np.zeros(2 * N)
        e[i] = h
        H[:, i] = (grad_l(u0 + e, prob) - grad_l(u0 - e, prob)) / (2 * h)
    H = 0.5 * (H + H.T)
    G = np.zeros((2 * N, 4))
    for c, pv in enumerate(param_values(prob, vr_n)):
        hp = h * max(1.0, abs(pv))
        G[:, c] = (grad_l(u0, with_param(prob, c, pv + hp, vr_n)) - grad_l(u0, with_param(prob, c, pv - hp, vr_n))) / (2 * hp)
    free = np.ones(2 * N, bool)
    for d in desc:
        if d[0] == "u":
            free[d[1]] = False
    hmax = max(1.0, float(np.abs(np.diag(H)[free]).max())) if free.any() else 1.0
    Z = scipy.linalg.null_space(A) if m else np.eye(2 * N)
    if Z.shape[1] and np.linalg.eigvalsh(Z.T @ H @ Z).min() <= SOSC_TOL * hmax:
        flags |= NOT_SOSC
    if flags & NAN_FLAGS:
        return nan_jac, flags, mu, res
    K = np.block([[H, A.T], [A, np.zeros((m, m))]])
    sol = np.linalg.solve(K, np.concatenate([-G, np.zeros((m, 4))]))
    return sol[:2].copy(), flags, mu, res
