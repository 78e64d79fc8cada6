"""FP64 primal-dual interior-point oracle on the reference's LITERAL multiple-shooting NLP  --  TEST INFRASTRUCTURE ONLY.

The reference hands its NLP to CasADi's `nlpsol('solver', 'ipopt', ...)` (agents/pure_mpc.py:285-300):
  z      = [vec(X) column-major (4(N+1)); vec(U) (2N)]                       pure_mpc.py:260
  f(z)   = 10 state + w_c control + w_d input_diff (+ archive terms)          pure_mpc.py:128-212
  g(z)   = [x_0 - s0; x_{k+1} - x_k - dt f(x_k, u_k)] = 0                      pure_mpc.py:249-257
  bounds on every variable                                                    pure_mpc.py:267-280
  z0     = [tile(s0, N+1); 0]                                                 pure_mpc.py:240-246
  options: ipopt.tol 1e-6, ipopt.max_iter 1000, everything else default       pure_mpc.py:291-296

casadi==3.6.6 (requirements.txt:4; bundles IPOPT 3.14 + MUMPS) is a third-party wheel that is absent from
/root/reference and not installable here, so this module RESTATES IPOPT's published algorithm
(A. Waechter, L. T. Biegler, "On the implementation of an interior-point filter line-search algorithm
for large-scale nonlinear programming", Math. Program. 106 (2006), sections 2-3) with IPOPT 3.14's default
option values, on dense FP64 linear algebra:
  * gradient-based objective/constraint scaling at the user's starting point (nlp_scaling_max_gradient 100)
  * bound relaxation 1e-8, starting point pushed into the bounds (bound_push = bound_frac = 0.01),
    bound multipliers 1, least-squares equality multipliers (dropped above constr_mult_init_max 1000)
  * monotone barrier update (mu_init 0.1, kappa_mu 0.2, theta_mu 1.5, kappa_eps 10), tau = max(0.99, 1-mu)
  * exact Lagrangian Hessian, inertia correction (delta_w sequence 1e-4, x100 / x8, /3; delta_c 1e-8 mu^1/4)
  * filter line search with switching condition / Armijo / sufficient decrease, second-order corrections
    (max_soc 4, kappa_soc 0.99), filter reset at every barrier update, kappa_sigma multiplier reset
  * termination on the scaled optimality error E_0 <= tol with IPOPT's s_d / s_c scaling (s_max 100)
NOT restated: the restoration phase (a problem that would enter it is reported with `restoration=True`
and finished by a Levenberg-damped feasibility step; counted in the fixtures), the watchdog, and MUMPS'
pivoting (inertia comes from a dense LDL^T here).

PARITY UNPINNED for the basin: nothing here was compared with a real IPOPT run.  It is the closest
achievable predictor of which local optimum the reference returns from its own cold start; the optimum it
reports is certified independently (mpc_oracle.kkt_residual, SLSQP warm-start confirmation).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import numpy as np
from scipy.linalg import ldl

import mpc_oracle as orc
from mpc_oracle import Problem, Solution, N_REF, WHEELBASE, REAR_RATIO

# ----------------------------------------------------------------------------------------
# NLP functions of the literal formulation
# ----------------------------------------------------------------------------------------
class LiteralNLP:
    """f, grad f, g, Jacobian, Lagrangian Hessian of agents/pure_mpc.py:128-280 for one Problem."""

    def __init__(self, prob: Problem):
        self.p = prob
        ref = prob.ref
        N = prob.N
        self.N, self.dt = N, prob.dt
        self.nx = 4 * (N + 1)
        self.n = self.nx + 2 * N
        self.m = self.nx
        j = np.minimum(prob.ego_index + np.arange(N), N_REF - 1)
        self.rx, self.ry, self.rh = ref[j, 0], ref[j, 1], ref[j, 3]
        self.sh, self.ch = np.sin(self.rh), np.cos(self.rh)
        self.obs = (orc.obstacle_positions(prob.others, N, prob.dt)
                    if (prob.others.shape[0] > 0 and prob.w_distance != 0.0 and not prob.literal_no_collision) else None)
        lo = np.tile([-orc.XY_MAX, -orc.XY_MAX, orc.TH_MIN, orc.V_MIN], N + 1)
        hi = np.tile([orc.XY_MAX, orc.XY_MAX, orc.TH_MAX, orc.V_MAX], N + 1)
        self.lb = np.concatenate([lo, np.tile([-orc.A_MAX, -orc.DELTA_MAX], N)])
        self.ub = np.concatenate([hi, np.tile([orc.A_MAX, orc.DELTA_MAX], N)])
        self.z0 = np.concatenate([np.tile(prob.s0, N + 1), np.zeros(2 * N)])

    def unpack(self, z):
        return z[:self.nx].reshape(self.N + 1, 4), z[self.nx:].reshape(self.N, 2)

    # ---- objective -----------------------------------------------------------------------
    def f(self, z) -> float:
        X, U = self.unpack(z)
        return orc.total_cost_from_components(orc.cost_components(X, U, self.p), self.p)

    def grad_hess_f(self, z, want_hess: bool):
        """gradient (n,) and, if asked, the dense Hessian (n, n) of the objective."""
        p, N, nx = self.p, self.N, self.nx
        X, U = self.unpack(z)
        g = np.zeros(self.n)
        H = np.zeros((self.n, self.n)) if want_hess else None
        gX = g[:nx].reshape(N + 1, 4)
        gU = g[nx:].reshape(N, 2)
        gU += p.w_control * 0.02 * U
        dU = np.diff(U, axis=0)
        gU[1:] += p.w_input_diff * 0.02 * dU
        gU[:-1] -= p.w_input_diff * 0.02 * dU
        if want_hess:
            for k in range(N):
                for i in range(2):
                    q = nx + 2 * k + i
                    H[q, q] += p.w_control * 0.02
                    if k > 0:
                        r = q - 2
                        H[q, q] += p.w_input_diff * 0.02
                        H[r, r] += p.w_input_diff * 0.02
                        H[q, r] -= p.w_input_diff * 0.02
                        H[r, q] -= p.w_input_diff * 0.02
        if not p.literal_no_collision:
            sh, ch = self.sh, self.ch
            dx, dy = X[:N, 0] - self.rx, X[:N, 1] - self.ry
            perp = dx * sh - dy * ch
            para = dx * ch + dy * sh
            gX[:N, 0] = 10 * (8 * perp * sh + 4 * para * ch)
            gX[:N, 1] = 10 * (-8 * perp * ch + 4 * para * sh)
            gX[:N, 2] = 10 * (X[:N, 2] - self.rh)
            gX[:N, 3] = 20 * p.w_speed * (X[:N, 3] - p.ref_v)
            hxx = 80 * sh * sh + 40 * ch * ch
            hxy = -40 * sh * ch
            hyy = 80 * ch * ch + 40 * sh * sh
            hvv = np.full(N, 20 * p.w_speed)
            if self.obs is not None:
                P = self.obs
                ex, ey = X[:N, None, 0] - P[:, :, 0], X[:N, None, 1] - P[:, :, 1]
                d = np.hypot(ex, ey)
                ds = np.maximum(d, 1e-300)
                cc = p.w_distance * np.where(d < 1.0, 1000.0, 100.0)
                f1 = -2.0 * cc / (d + 1e-6) ** 3            # phi'(d)
                f2 = 6.0 * cc / (d + 1e-6) ** 4             # phi''(d)
                nxv, nyv = ex / ds, ey / ds
                gX[:N, 0] += np.sum(f1 * nxv, axis=1)
                gX[:N, 1] += np.sum(f1 * nyv, axis=1)
                tang = f1 / ds
                rad = f2 - tang
                hxx = hxx + np.sum(rad * nxv * nxv + tang, axis=1)
                hxy = hxy + np.sum(rad * nxv * nyv, axis=1)
                hyy = hyy + np.sum(rad * nyv * nyv + tang, axis=1)
            if p.w_collision != 0.0 and p.is_collide:
                gX[:N, 3] += p.w_collision * 6000.0 * X[:N, 3]
                hvv = hvv + p.w_collision * 6000.0
            if want_hess:
                for k in range(N):
                    o = 4 * k
                    H[o, o] += hxx[k]; H[o, o + 1] += hxy[k]; H[o + 1, o] += hxy[k]; H[o + 1, o + 1] += hyy[k]
                    H[o + 2, o + 2] += 10.0
                    H[o + 3, o + 3] += hvv[k]
        return g, H

    # ---- constraints ---------------------------------------------------------------------
    def _dyn_terms(self, X, U):
        N = self.N
        th, v, dl = X[:N, 2], X[:N, 3], U[:, 1]
        t = np.tan(dl)
        beta = np.arctan(REAR_RATIO * t)
        q = 1 + REAR_RATIO * REAR_RATIO * t * t
        b1 = REAR_RATIO * (1 + t * t) / q                                   # beta'
        b2 = (2 * REAR_RATIO * (1 - REAR_RATIO ** 2)) * t * (1 + t * t) / (q * q)   # beta'' (= 0.75 t (1+t^2)/q^2)
        c, s = np.cos(th + beta), np.sin(th + beta)
        return th, v, beta, b1, b2, c, s

    def g(self, z):
        X, U = self.unpack(z)
        N, dt = self.N, self.dt
        th, v, beta, b1, b2, c, s = self._dyn_terms(X, U)
        r = np.empty((N + 1, 4))
        r[0] = X[0] - self.p.s0
        r[1:, 0] = X[1:, 0] - (X[:N, 0] + dt * v * c)
        r[1:, 1] = X[1:, 1] - (X[:N, 1] + dt * v * s)
        r[1:, 2] = X[1:, 2] - (X[:N, 2] + dt * (v / WHEELBASE) * np.sin(beta))
        r[1:, 3] = X[1:, 3] - (X[:N, 3] + dt * U[:, 0])
        return r.reshape(-1)

    def jac(self, z):
        X, U = self.unpack(z)
        N, dt, nx = self.N, self.dt, self.nx
        th, v, beta, b1, b2, c, s = self._dyn_terms(X, U)
        J = np.zeros((self.m, self.n))
        J[np.arange(self.m), np.arange(self.m)] = 1.0
        for k in range(N):
            r0, c0, u0 = 4 * (k + 1), 4 * k, nx + 2 * k
            J[r0 + 0, c0 + 0] = -1; J[r0 + 0, c0 + 2] = dt * v[k] * s[k]; J[r0 + 0, c0 + 3] = -dt * c[k]
            J[r0 + 1, c0 + 1] = -1; J[r0 + 1, c0 + 2] = -dt * v[k] * c[k]; J[r0 + 1, c0 + 3] = -dt * s[k]
            J[r0 + 2, c0 + 2] = -1; J[r0 + 2, c0 + 3] = -dt * math.sin(beta[k]) / WHEELBASE
            J[r0 + 3, c0 + 3] = -1
            J[r0 + 0, u0 + 1] = dt * v[k] * s[k] * b1[k]
            J[r0 + 1, u0 + 1] = -dt * v[k] * c[k] * b1[k]
            J[r0 + 2, u0 + 1] = -dt * (v[k] / WHEELBASE) * math.cos(beta[k]) * b1[k]
            J[r0 + 3, u0 + 0] = -dt
        return J

    def hess_lag(self, z, lam, sigma_f: float):
        """sigma_f * Hess f + sum_i lam_i Hess g_i (dense)."""
        _, H = self.grad_hess_f(z, True)
        H *= sigma_f
        X, U = self.unpack(z)
        N, dt, nx = self.N, self.dt, self.nx
        th, v, beta, b1, b2, c, s = self._dyn_terms(X, U)
        L = lam.reshape(N + 1, 4)
        cb, sb = np.cos(beta), np.sin(beta)
        for k in range(N):
            l1, l2, l3 = L[k + 1, 0], L[k + 1, 1], L[k + 1, 2]
            # second derivatives of -dt f_dyn in (theta, v, delta)
            ck, sk, vk, g1, g2 = c[k], s[k], v[k], b1[k], b2[k]
            hthth = -dt * (l1 * (-vk * ck) + l2 * (-vk * sk))
            hthv = -dt * (l1 * (-sk) + l2 * ck)
            hthd = -dt * (l1 * (-vk * ck * g1) + l2 * (-vk * sk * g1))
            hvd = -dt * (l1 * (-sk * g1) + l2 * (ck * g1) + l3 * (cb[k] * g1 / WHEELBASE))
            hdd = -dt * (l1 * (-vk * ck * g1 * g1 - vk * sk * g2) + l2 * (-vk * sk * g1 * g1 + vk * ck * g2)
                         + l3 * (vk / WHEELBASE) * (-sb[k] * g1 * g1 + cb[k] * g2))
            it, iv, idl = 4 * k + 2, 4 * k + 3, nx + 2 * k + 1
            H[it, it] += hthth
            H[it, iv] += hthv; H[iv, it] += hthv
            H[it, idl] += hthd; H[idl, it] += hthd
            H[iv, idl] += hvd; H[idl, iv] += hvd
            H[idl, idl] += hdd
        return H


# ----------------------------------------------------------------------------------------
# IPOPT's algorithm (Waechter & Biegler 2006), default options of IPOPT 3.14
# ----------------------------------------------------------------------------------------
@dataclass
class IpoptOptions:
    tol: float = 1e-6                     # pure_mpc.py:295
    max_iter: int = 1000                  # pure_mpc.py:294
    dual_inf_tol: float = 1.0
    constr_viol_tol: float = 1e-4
    compl_inf_tol: float = 1e-4
    mu_init: float = 0.1
    kappa_mu: float = 0.2                 # mu_linear_decrease_factor
    theta_mu: float = 1.5                 # mu_superlinear_decrease_power
    kappa_eps: float = 10.0               # barrier_tol_factor
    tau_min: float = 0.99
    bound_push: float = 0.01
    bound_frac: float = 0.01
    bound_relax_factor: float = 1e-8
    bound_mult_init_val: float = 1.0
    constr_mult_init_max: float = 1000.0
    nlp_scaling_max_gradient: float = 100.0
    s_max: float = 100.0
    kappa_sigma: float = 1e10
    # line search
    eta_phi: float = 1e-8
    gamma_theta: float = 1e-5
    gamma_phi: float = 1e-8
    delta: float = 1.0
    s_phi: float = 2.3
    s_theta: float = 1.1
    theta_min_fact: float = 1e-4
    theta_max_fact: float = 1e4
    alpha_min_frac: float = 0.05
    alpha_red_factor: float = 0.5
    max_soc: int = 4
    kappa_soc: float = 0.99
    # inertia correction
    delta_w_init: float = 1e-4            # first_hessian_perturbation
    delta_w_min: float = 1e-20
    delta_w_max: float = 1e20
    kappa_w_minus: float = 1.0 / 3.0
    kappa_w_plus: float = 8.0
    kappa_w_plus_first: float = 100.0
    delta_c_bar: float = 1e-8             # jacobian_regularization_value
    kappa_c: float = 0.25


@dataclass
class IpmResult:
    z: np.ndarray
    U: np.ndarray
    X: np.ndarray
    cost: float                  # objective of the ROLLOUT of U (what applying U gives), like mpc_oracle.Solution.cost
    f_nlp: float                 # objective at the NLP iterate z
    success: bool
    iters: int
    status: str
    restoration: bool
    constr_viol: float
    mu: float

    @property
    def u0(self) -> np.ndarray:
        return self.U[0].copy()


def _inertia_solve(K: np.ndarray, rhs: np.ndarray, n: int, m: int):
    """Dense symmetric-indefinite solve; returns (solution or None, n_neg, singular).  The matrix is
    equilibrated symmetrically first (inertia is invariant under congruence; Sigma spans 1e-10..1e+10)."""
    d = 1.0 / np.sqrt(np.maximum(np.max(np.abs(K), axis=1), 1e-300))
    Ks = K * d[:, None] * d[None, :]
    try:
        L, D, perm = ldl(Ks, lower=True, hermitian=True)
    except Exception:
        return None, -1, True
    ev = []
    i, nk = 0, K.shape[0]
    while i < nk:
        if i + 1 < nk and D[i + 1, i] != 0.0:
            a, b, c = D[i, i], D[i + 1, i], D[i + 1, i + 1]
            tr, det = a + c, a * c - b * b
            disc = math.sqrt(max(tr * tr / 4 - det, 0.0))
            ev += [tr / 2 - disc, tr / 2 + disc]
            i += 2
        else:
            ev.append(D[i, i])
            i += 1
    ev = np.array(ev)
    if not np.all(np.isfinite(ev)):
        return None, -1, True
    zero = int(np.sum(np.abs(ev) <= 1e-13))
    neg = int(np.sum(ev < -1e-13))
    if zero > 0:
        return None, neg, True
    if neg != m:
        return None, neg, False
    sol = d * np.linalg.solve(Ks, d * rhs)
    return sol, neg, False


def solve_ipopt_like(prob: Problem, opts: Optional[IpoptOptions] = None, trace: bool = False) -> IpmResult:
    o = opts or IpoptOptions()
    nlp = LiteralNLP(prob)
    n, m = nlp.n, nlp.m
    # ---- scaling at the user's starting point (gradient-based)
    g0, _ = nlp.grad_hess_f(nlp.z0, False)
    gmax = float(np.max(np.abs(g0)))
    sf = o.nlp_scaling_max_gradient / gmax if gmax > o.nlp_scaling_max_gradient else 1.0
    sf = max(sf, 1e-8)
    J0 = nlp.jac(nlp.z0)
    rmax = np.max(np.abs(J0), axis=1)
    sc = np.where(rmax > o.nlp_scaling_max_gradient, o.nlp_scaling_max_gradient / np.maximum(rmax, 1e-300), 1.0)
    sc = np.maximum(sc, 1e-8)
    # ---- relaxed bounds, interior starting point
    lb = nlp.lb - o.bound_relax_factor * np.maximum(1.0, np.abs(nlp.lb))
    ub = nlp.ub + o.bound_relax_factor * np.maximum(1.0, np.abs(nlp.ub))
    pl = np.minimum(o.bound_push * np.maximum(1.0, np.abs(lb)), o.bound_frac * (ub - lb))
    pu = np.minimum(o.bound_push * np.maximum(1.0, np.abs(ub)), o.bound_frac * (ub - lb))
    x = np.minimum(np.maximum(nlp.z0, lb + pl), ub - pu)
    zl = np.full(n, o.bound_mult_init_val)
    zu = np.full(n, o.bound_mult_init_val)

    def fs(xx):
        return sf * nlp.f(xx)

    def cs(xx):
        return sc * nlp.g(xx)

    def grads(xx):
        g, _ = nlp.grad_hess_f(xx, False)
        return sf * g

    def jacs(xx):
        return sc[:, None] * nlp.jac(xx)

    # least-squares multipliers
    gf = grads(x)
    J = jacs(x)
    K = np.zeros((n + m, n + m))
    K[:n, :n] = np.eye(n)
    K[:n, n:] = J.T
    K[n:, :n] = J
    try:
        sol = np.linalg.solve(K, -np.concatenate([gf - zl + zu, np.zeros(m)]))
        lam = sol[n:]
        if np.max(np.abs(lam)) > o.constr_mult_init_max:
            lam = np.zeros(m)
    except np.linalg.LinAlgError:
        lam = np.zeros(m)

    mu = o.mu_init
    tau = max(o.tau_min, 1.0 - mu)
    filt = []
    c = cs(x)
    theta0 = float(np.sum(np.abs(c)))
    theta_min = o.theta_min_fact * max(1.0, theta0)
    theta_max = o.theta_max_fact * max(1.0, theta0)
    delta_w_last = 0.0
    status, restoration = "max_iter", False
    it = 0

    def barrier(xx, mu_):
        sl, su = xx - lb, ub - xx
        if np.any(sl <= 0) or np.any(su <= 0):
            return math.inf
        return fs(xx) - mu_ * (np.sum(np.log(sl)) + np.sum(np.log(su)))

    def err(mu_, gf_, J_, c_, lam_, zl_, zu_, x_):
        sl, su = x_ - lb, ub - x_
        sd = max(o.s_max, (np.sum(np.abs(lam_)) + np.sum(np.abs(zl_)) + np.sum(np.abs(zu_))) / (m + 2 * n)) / o.s_max
        sc_ = max(o.s_max, (np.sum(np.abs(zl_)) + np.sum(np.abs(zu_))) / (2 * n)) / o.s_max
        dual = float(np.max(np.abs(gf_ + J_.T @ lam_ - zl_ + zu_)))
        prim = float(np.max(np.abs(c_)))
        comp = float(max(np.max(np.abs(sl * zl_ - mu_)), np.max(np.abs(su * zu_ - mu_))))
        return max(dual / sd, prim, comp / sc_), dual, prim, comp

    tiny_count = 0
    while it < o.max_iter:
        gf = grads(x)
        J = jacs(x)
        c = cs(x)
        E0, dual, prim, comp0 = err(0.0, gf, J, c, lam, zl, zu, x)
        if (E0 <= o.tol and dual / sf <= o.dual_inf_tol and float(np.max(np.abs(c / sc))) <= o.constr_viol_tol
                and comp0 / sf <= o.compl_inf_tol):
            status = "success"
            break
        # ---- barrier update (possibly several times)
        while True:
            Emu = err(mu, gf, J, c, lam, zl, zu, x)[0]
            if Emu <= o.kappa_eps * mu and mu > o.tol / 10.0 * (1 + 1e-12):
                mu = max(o.tol / 10.0, min(o.kappa_mu * mu, mu ** o.theta_mu))
                tau = max(o.tau_min, 1.0 - mu)
                filt = []
            else:
                break
        sl, su = x - lb, ub - x
        Sigma = zl / sl + zu / su
        W = nlp.hess_lag(x, lam * sc, sf)          # scaled Lagrangian: sf f + lam^T (sc g)
        gphi = gf - mu / sl + mu / su
        rhs = -np.concatenate([gphi + J.T @ lam, c])
        # ---- inertia correction
        dw, dc = 0.0, 0.0
        sol = None
        K = np.zeros((n + m, n + m))
        K[:n, n:] = J.T
        K[n:, :n] = J
        first_try = True
        while True:
            K[:n, :n] = W + np.diag(Sigma + dw)
            K[n:, n:] = -dc * np.eye(m)
            sol, neg, singular = _inertia_solve(K, rhs, n, m)
            if sol is not None:
                if dw > 0:
                    delta_w_last = dw
                break
            if singular and dc == 0.0:
                dc = o.delta_c_bar * mu ** o.kappa_c
            if first_try:
                first_try = False
                dw = o.delta_w_init if delta_w_last == 0.0 else max(o.delta_w_min, o.kappa_w_minus * delta_w_last)
            else:
                dw = dw * (o.kappa_w_plus_first if delta_w_last == 0.0 else o.kappa_w_plus)
            if dw > o.delta_w_max:
                break
        if sol is None:
            status, restoration = "inertia_failure", True
            break
        dx, dlam = sol[:n], sol[n:]
        dzl = mu / sl - zl - (zl / sl) * dx
        dzu = mu / su - zu + (zu / su) * dx

        def ftb(v, dv):
            neg_ = dv < 0
            if not np.any(neg_):
                return 1.0
            return float(min(1.0, np.min(-tau * v[neg_] / dv[neg_])))

        a_max = min(ftb(sl, dx), ftb(su, -dx))
        a_z = min(ftb(zl, dzl), ftb(zu, dzu))
        # ---- tiny step
        if float(np.max(np.abs(dx) / (1.0 + np.abs(x)))) < 10 * np.finfo(float).eps:
            tiny_count += 1
            x = x + a_max * dx
            lam = lam + a_max * dlam
            zl, zu = zl + a_z * dzl, zu + a_z * dzu
            it += 1
            if tiny_count >= 2:
                if mu <= o.tol / 10.0 * (1 + 1e-12):
                    status = "tiny_step"
                    break
                mu = max(o.tol / 10.0, min(o.kappa_mu * mu, mu ** o.theta_mu))
                tau = max(o.tau_min, 1.0 - mu)
                filt = []
                tiny_count = 0
            continue
        tiny_count = 0
        # ---- filter line search
        theta = float(np.sum(np.abs(c)))
        phi = barrier(x, mu)
        dphi = float(gphi @ dx)
        if dphi < 0 and theta <= theta_min:
            a_min = min(o.gamma_theta, o.gamma_phi * theta / (-dphi) if theta > 0 else math.inf,
                        o.delta * theta ** o.s_theta / (-dphi) ** o.s_phi if theta > 0 else math.inf)
        elif dphi < 0:
            a_min = min(o.gamma_theta, o.gamma_phi * theta / (-dphi))
        else:
            a_min = o.gamma_theta
        a_min *= o.alpha_min_frac

        def in_filter(th_, ph_):
            return any(th_ >= tf and ph_ >= pf for tf, pf in filt)

        def switching(a_):
            return dphi < 0 and a_ * (-dphi) ** o.s_phi > o.delta * theta ** o.s_theta

        def acceptable(th_t, ph_t, a_test):
            if not (th_t <= theta_max) or not math.isfinite(ph_t):
                return False, False
            if in_filter(th_t, ph_t):
                return False, False
            if theta <= theta_min and switching(a_test):
                okk = ph_t <= phi + o.eta_phi * a_test * dphi + 10 * np.finfo(float).eps * abs(phi)
                return okk, True
            okk = th_t <= (1 - o.gamma_theta) * theta or ph_t <= phi - o.gamma_phi * theta
            return okk, False

        a = a_max
        accepted = False
        x_new = None
        ftype = False
        first = True
        while a >= a_min:
            xt = x + a * dx
            ct = cs(xt)
            th_t = float(np.sum(np.abs(ct)))
            ph_t = barrier(xt, mu)
            okk, ft = acceptable(th_t, ph_t, a)
            if okk:
                accepted, x_new, ftype = True, xt, ft
                break
            # second-order correction on the first trial step
            if first and th_t >= theta and o.max_soc > 0:
                c_soc = a * c + ct
                th_old = theta
                for _ in range(o.max_soc):
                    rhs_soc = -np.concatenate([gphi + J.T @ lam, c_soc])
                    s2 = np.linalg.solve(K, rhs_soc)
                    dxs = s2[:n]
                    a_soc = min(ftb(sl, dxs), ftb(su, -dxs))
                    xs = x + a_soc * dxs
                    cst = cs(xs)
                    th_s = float(np.sum(np.abs(cst)))
                    ph_s = barrier(xs, mu)
                    oks, fts = acceptable(th_s, ph_s, a)
                    if oks:
                        accepted, x_new, ftype = True, xs, fts
                        dlam = s2[n:]
                        # bound multipliers follow the corrected primal step
                        dzl = mu / sl - zl - (zl / sl) * dxs
                        dzu = mu / su - zu + (zu / su) * dxs
                        a_z = min(ftb(zl, dzl), ftb(zu, dzu))
                        a = a_soc
                        break
                    if th_s > o.kappa_soc * th_old:
                        break
                    c_soc = a_soc * c_soc + cst
                    th_old = th_s
                if accepted:
                    break
            first = False
            a *= o.alpha_red_factor
        if not accepted:
            # IPOPT would enter the restoration phase here (not restated): take a damped feasibility
            # (Gauss-Newton on ||c||^2 with the barrier Hessian as metric) step instead and flag the run
            restoration = True
            Kr = np.zeros((n + m, n + m))
            Kr[:n, :n] = np.diag(Sigma + 1.0)
            Kr[:n, n:] = J.T
            Kr[n:, :n] = J
            Kr[n:, n:] = -1e-8 * np.eye(m)
            sr = np.linalg.solve(Kr, -np.concatenate([np.zeros(n), c]))
            dxr = sr[:n]
            ar = min(ftb(sl, dxr), ftb(su, -dxr))
            done_r = False
            while ar > 1e-12:
                xt = x + ar * dxr
                if float(np.sum(np.abs(cs(xt)))) < (1 - 1e-4 * ar) * theta:
                    x = xt
                    done_r = True
                    break
                ar *= 0.5
            if not done_r:
                status = "restoration_failed"
                break
            filt.append(((1 - o.gamma_theta) * theta, phi - o.gamma_phi * theta))
            it += 1
            continue
        # ---- filter augmentation (when the step was not an f-type step with Armijo)
        if not (ftype and theta <= theta_min):
            filt.append(((1 - o.gamma_theta) * theta, phi - o.gamma_phi * theta))
        x = x_new
        lam = lam + a * dlam
        zl = zl + a_z * dzl
        zu = zu + a_z * dzu
        sl, su = x - lb, ub - x
        zl = np.maximum(np.minimum(zl, o.kappa_sigma * mu / sl), mu / (o.kappa_sigma * sl))
        zu = np.maximum(np.minimum(zu, o.kappa_sigma * mu / su), mu / (o.kappa_sigma * su))
        it += 1
        if trace:
            print(f"it {it:3d} f {fs(x) / sf:.8g} theta {float(np.sum(np.abs(cs(x)))):.3e} mu {mu:.2e} a {a:.3g} az {a_z:.3g} dw {dw:.2e}")

    X, U = nlp.unpack(x)
    U = np.clip(U, [-orc.A_MAX, -orc.DELTA_MAX], [orc.A_MAX, orc.DELTA_MAX])
    Xr = orc.rollout(prob.s0, U, prob.dt)
    comp = orc.cost_components(Xr, U, prob)
    return IpmResult(z=x.copy(), U=U.copy(), X=Xr, cost=float(orc.total_cost_from_components(comp, prob)),
                     f_nlp=float(nlp.f(x)), success=(status == "success"), iters=it, status=status,
                     restoration=restoration, constr_viol=float(np.max(np.abs(nlp.g(x)))), mu=mu)


def polish(prob: Problem, U: np.ndarray) -> Solution:
    """SLSQP (single shooting) started at U: removes the O(mu) distance an interior-point iterate keeps from
    active bounds.  Used to report `best(IPM basin, polished)`."""
    return orc.solve_nlp(prob, U0=U)


# ----------------------------------------------------------------------------------------
# best known optimum of one problem: portfolio of the two CPU solvers + fixed-point polish
# ----------------------------------------------------------------------------------------
def polish_fixed_point(prob: Problem, U: np.ndarray, rounds: int = 4, du_tol: float = 1e-3, gain_tol: float = 1e-6,
                       viol_tol: float = 1e-3):
    """Repeats SLSQP (single shooting, started at the candidate) until a run neither moves the first
    control by `du_tol` nor lowers the cost by `gain_tol` relative -- the 'oracle confirms it' criterion of
    the parity tests, applied to the oracle's own candidates.  Every SLSQP result is first pulled back into the
    feasible set (mpc_oracle.repair_feasible): SLSQP satisfies the node bounds only to its tolerance, and a failed run
    can return a grossly infeasible point that would otherwise look like a fixed point with a low cost; a result
    that violates a bound by more than `viol_tol` is rejected.  Returns (U, cost, confirmed) with U feasible."""
    U = orc.repair_feasible(np.asarray(U, dtype=np.float64), prob)
    c = orc.objective(U, prob)
    for _ in range(rounds):
        s = orc.solve_nlp(prob, U0=U)
        if orc.bound_violation(s.U, prob) > viol_tol:
            return U, c, False                       # SLSQP failed into the infeasible region
        Un = orc.repair_feasible(s.U, prob)
        cn = orc.objective(Un, prob)
        if not np.isfinite(cn) or cn > c + 1e-9 * (1 + abs(c)):
            # no feasible improvement: a fixed point if SLSQP did not move either
            du0 = float(np.max(np.abs(Un[0] - U[0])))
            return U, c, bool(np.isfinite(cn) and du0 < du_tol and cn <= c + gain_tol * (1 + abs(c)))
        du0 = float(np.max(np.abs(Un[0] - U[0])))
        gain = (c - cn) / (1.0 + abs(c))
        U, c = Un, cn
        if du0 < du_tol and gain < gain_tol:
            return U, c, True
    return U, c, False


# the starts of the CPU portfolio behind the yardstick: zero controls plus constant-acceleration / steering-pulse
# perturbations (a, delta, stages the pulse lasts).  They were the device solver's table when the fixtures were generated;
# the device's table (mpc_core.cuh: start_controls) has since been re-selected on a separate tuning set, the yardstick's
# starts stay fixed so that the committed fixtures stay valid.
PORTFOLIO_STARTS = ((0.0, 0.0, 0), (-5.0, 0.0, 0), (0.0, -0.9, 3), (0.0, 0.4, 3), (5.0, 0.9, 3), (0.0, -0.4, 3), (0.0, -0.4, 1 << 20), (5.0, -0.4, 3))


def start_controls(st: int, N: int) -> np.ndarray:
    a, d, nk = PORTFOLIO_STARTS[st]
    U = np.zeros((N, 2))
    U[:, 0] = a
    U[: min(nk, N), 1] = d
    return U


def path_following_controls(prob: Problem, mode: str = "ref", look: int = 1, slalom: bool = False) -> np.ndarray:
    """What a driver would do, as an initial guess: roll the model of pure_mpc.py:220-228 / 252-254 forward steering at
    the path point `look` rows ahead of the stage's own (pure_mpc.py:129 indexing: min(ego_index + k + look, 84)) with the
    steering angle that turns the heading onto it within the step, and with the acceleration that reaches the stage's
    reference speed within the step (`mode` "ref") or full braking ("brake"), inside the bounds of :272-280.
    `slalom`: from the first stage whose reference row is the frozen last row of the path (k >= 84 - ego_index) the
    steering alternates full right / full left every stage -- the shape of the optima past the end of the path.
    The device solver's path-following starts (mpc_core.cuh: apply_start) follow the same recipe in FP32."""
    ref = prob.ref
    sb_max = math.sin(math.atan(orc.REAR_RATIO * math.tan(orc.DELTA_MAX)))
    U = np.zeros((prob.N, 2))
    s = np.asarray(prob.s0, dtype=np.float64).copy()
    for k in range(prob.N):
        j = min(prob.ego_index + k + look, ref.shape[0] - 1)
        a = -orc.A_MAX if mode == "brake" else (prob.ref_v[min(k, len(prob.ref_v) - 1)] - s[3]) / prob.dt
        a = min(max(a, -orc.A_MAX), orc.A_MAX)
        a = min(max(a, (orc.V_MIN - s[3]) / prob.dt), (orc.V_MAX - s[3]) / prob.dt)
        ex, ey = ref[j, 0] - s[0], ref[j, 1] - s[1]
        des = math.atan2(ey, ex) if ex * ex + ey * ey > 1e-6 else ref[j, 3]
        dth = math.atan2(math.sin(des - s[2]), math.cos(des - s[2]))
        sb = min(max(dth / (prob.dt * max(s[3], 1e-3) / orc.WHEELBASE), -sb_max), sb_max)
        k_end = ref.shape[0] - 1 - prob.ego_index
        if slalom and k >= k_end:
            sb = sb_max if (k - k_end) & 1 else -sb_max
        U[k] = (a, math.asin(min(max(sb / math.sqrt(0.25 + 0.75 * sb * sb), -1.0), 1.0)))
        s = orc.step(s, U[k], prob.dt)
    return orc.repair_feasible(U, prob)


def best_known_optimum(prob: Problem, cpu_starts: int = 4, path_starts: int = 2):
    """The yardstick of the solve-parity tests: the lowest-cost CONFIRMED local optimum found by
    (a) the IPOPT-like interior point on the literal multiple-shooting NLP from the reference's cold start,
    (b) SLSQP on the single-shooting form from zero controls (the reference's cold start in that form),
    (c) SLSQP from `cpu_starts - 1` perturbed starts (PORTFOLIO_STARTS), and
    (d) SLSQP from `path_starts` path-following starts (reference speed, full braking) -- the kind of start that turned
        out to reach the lowest optimum most often -- and, when the horizon runs past the end of the path, from the slalom
        start,
    so that a first-control disagreement means the device found a different optimum than EVERY one of seven (eight) CPU runs,
    not merely a better one than a single cold start; each candidate is polished to a feasible fixed point.  Returns a dict
    with the winner and the candidates."""
    r = solve_ipopt_like(prob)
    Ui, ci, oki = polish_fixed_point(prob, r.U)
    s = orc.solve_nlp(prob)
    Us, cs, oks = polish_fixed_point(prob, s.U)
    cands = [("ipm", Ui, ci, oki), ("slsqp", Us, cs, oks)]
    for st in range(1, cpu_starts):
        sk = orc.solve_nlp(prob, U0=start_controls(st, prob.N))
        Uk, ck, okk = polish_fixed_point(prob, sk.U)
        cands.append((f"slsqp_start{st}", Uk, ck, okk))
    for mode in ("ref", "brake")[:path_starts]:
        sk = orc.solve_nlp(prob, U0=path_following_controls(prob, mode))
        Uk, ck, okk = polish_fixed_point(prob, sk.U)
        cands.append((f"slsqp_path_{mode}", Uk, ck, okk))
    if path_starts and prob.ego_index + prob.N > prob.ref.shape[0] - 1:
        sk = orc.solve_nlp(prob, U0=path_following_controls(prob, "ref", 1, slalom=True))
        Uk, ck, okk = polish_fixed_point(prob, sk.U)
        cands.append(("slsqp_slalom", Uk, ck, okk))
    conf = [c for c in cands if c[3]] or cands
    src, Ub, cb, okb = min(conf, key=lambda c: c[2])
    return dict(U=Ub, cost=cb, success=okb, source=src,
                ipm_U=Ui, ipm_cost=ci, ipm_confirmed=oki, ipm_raw_U=r.U, ipm_raw_cost=r.cost, ipm_status=r.status,
                ipm_restoration=r.restoration, ipm_iters=r.iters,
                slsqp_U=Us, slsqp_cost=cs, slsqp_confirmed=oks)
