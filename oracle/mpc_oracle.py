"""FP64 CPU oracle for the PureMPC_Agent hot path  --  TEST INFRASTRUCTURE ONLY.

This module restates, in numpy/scipy double precision, the algorithm of the
reference's per-step MPC (SaeedRahmani/MPC-RL_for_AVs).  It is the *checker* for the
CUDA path.  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU legs may
import it; the product package must never route through it.

PARITY: PINNED TO THE REFERENCE'S OWN CODE EXCEPT FOR TWO THIRD-PARTY PRIMITIVES.
The reference holds no golden vectors, known-answer tests or fixtures for this path (its test_*.py
are GUI demos), and its two native dependencies are absent and not installable here:
``casadi==3.6.6`` (SX graph + IPOPT/MUMPS; requirements.txt:4) and ``shapely==2.0.6`` (GEOS;
requirements.txt:7).  What was done instead (tests/golden/make_reference_golden.py ->
tests/golden/golden_reference.npz, checked by tests/test_reference_pin.py):
the UNMODIFIED agents/pure_mpc.py, agents/pure_mpc_no_collision.py and agents/archive/pure_mpc.py are
imported from /root/reference
and executed with numeric stand-ins for casadi (numbers instead of symbols: every cost / constraint
expression is evaluated by the reference's own lines at an injected trajectory) and shapely (textbook
segment intersection).  Against those outputs this module is
  * exact on every discrete output: nearest path index, per-vehicle collision flags, conflict indices,
    is_collide, the 10-step latch over 16-step sequences (192 scenes + 24 x 16 sequence steps, 0 mismatches);
  * within 4e-8 relative on the shipped objective and its components, 2e-6 on parsed state and
    regenerated speeds, 1.3e-4 relative on the archive's obstacle-distance term -- all of it one
    quirk (Q11): under the reference's pinned numpy 2.x, np.float32 scalars stay float32 against
    Python floats (NEP 50), so the reference carries the ego speed, a wrapped heading and the other
    vehicles' in-NLP predicted positions in float32; this module uses float64 on the exact float32 inputs
    (what the same reference computes under numpy 1.x promotion).  The one place where that choice would
    change a DISCRETE output is kept in float32 like the reference: the other vehicles' 31-point tracks of
    the collision check (predict_other_polyline), where float32 accumulation keeps a same-lane vehicle
    exactly on the path's line;
  * identical bounds, cold start and dynamics constraints (the rollout below zeroes the reference's g).
STILL UNPINNED: GEOS' intersection primitive (incl. the order of MultiPoint members: assumed
lexicographic) and which local optimum IPOPT returns from the cold start.  For the latter the NLP is
solved here by an independent method (scipy SLSQP on the single-shooting form; the literal
multiple-shooting form of pure_mpc.py:230-300 is provided for cross-checks) with a
solver-independent KKT certificate (`kkt_residual`).

State order [x, y, theta, v], control order [a, delta]  (agents/pure_mpc.py:88-89).
"""
from __future__ import annotations

import functools
import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

# ----------------------------------------------------------------------------------------
# constants (reference file:line in comments)
# ----------------------------------------------------------------------------------------
WHEELBASE = 2.5                      # agents/utils.py:18
REAR_RATIO = 0.5                     # LENGTH_REAR / LENGTH, agents/utils.py:19
MAX_ACCEL_PRED = 3.5                 # Vehicle.max_acceleration, agents/utils.py:39
A_MAX = 5.0                          # agents/pure_mpc.py:279-280
DELTA_MAX = math.pi / 3.0            # agents/pure_mpc.py:279-280
V_MIN, V_MAX = 0.0, 30.0             # agents/pure_mpc.py:273-274
TH_MIN, TH_MAX = -math.pi, math.pi   # agents/pure_mpc.py:273-274
XY_MAX = 500.0                       # agents/pure_mpc.py:273-274
N_REF = 85                           # 40 + 20 + 25 rows, agents/base_agent.py:127-152
PRED_HORIZON = 30                    # agents/pure_mpc.py:554
TIME_THRESHOLD = 30                  # agents/pure_mpc.py:555
SAFETY_BUFFER_POINTS = 5             # agents/pure_mpc.py:681
MEMORY_STEPS = 10                    # agents/pure_mpc.py:39
COLLIDE_SPEED_WEIGHT = 100.0         # agents/pure_mpc.py:144-147


def reference_states(dt: float = 0.1) -> np.ndarray:
    """The hard-coded left-turn path, (85, 4) rows (x, y, v, heading).

    Follows agents/base_agent.py:118-154: start (2, 50), v = 10; 40 straight steps with
    heading -pi/2; 20 turn steps, heading decremented by (pi/2)/20 *before* each move;
    25 straight steps that only advance x.  The arithmetic order of the original
    accumulation is kept so the table is bit-identical in FP64.
    """
    x, y, v, h = 2.0, 50.0, 10.0, -np.pi / 2
    rows = []
    for _ in range(40):
        x += 0
        y += v * dt * np.sin(h)
        rows.append((x, y, v, h))
    step = (np.pi / 2) / 20
    for _ in range(20):
        h -= step
        x += v * dt * np.cos(h)
        y += v * dt * np.sin(h)
        rows.append((x, y, v, h))
    for _ in range(25):
        x += v * dt * np.cos(h)
        y += 0
        rows.append((x, y, v, h))
    return np.array(rows, dtype=np.float64)


@functools.lru_cache(maxsize=None)
def path_table(dt: float = 0.1) -> np.ndarray:
    """reference_states(dt), computed once per dt and read-only: the table every function below takes from
    `Problem.ref` or from its own dt."""
    t = reference_states(dt)
    t.setflags(write=False)
    return t


def normalize_angle(angle: float) -> float:
    """Wrap to [-pi, pi] by repeated +-2pi (agents/base_agent.py:156-170)."""
    angle = float(angle)
    while angle > np.pi:
        angle -= 2 * np.pi
    while angle < -np.pi:
        angle += 2 * np.pi
    return angle


@dataclass
class ParsedObs:
    ego: np.ndarray                 # (4,) x, y, theta(wrapped), speed
    others: np.ndarray              # (n, 4) x, y, speed, heading (NOT wrapped)


def parse_obs(obs: np.ndarray, vehicles_count: Optional[int] = None) -> ParsedObs:
    """agents/base_agent.py:81-116.  Row 0 is the ego; rows 1..n the present others,
    n = (number of rows with presence == 1) - 1; speed = ||(vx, vy)|| (agents/utils.py:36)."""
    if not isinstance(obs, np.ndarray):
        raise TypeError(f"Expect observation type np.ndarray, but got {type(obs)}.")
    if vehicles_count is not None and obs.shape != (vehicles_count, 8):
        raise ValueError(f"Expect observation's shape of ({(vehicles_count, 8)}), but got {obs.shape}")
    o = obs.astype(np.float64)
    n = int(np.sum(obs[:, 0] == 1)) - 1
    ego = np.array([o[0, 1], o[0, 2], normalize_angle(o[0, 5]), float(_norm2(o[0, 3], o[0, 4]))])
    others = np.zeros((max(n, 0), 4))
    for i in range(max(n, 0)):
        r = o[i + 1]
        others[i] = (r[1], r[2], float(_norm2(r[3], r[4])), r[5])
    return ParsedObs(ego=ego, others=others)


def _norm2(dx, dy):
    """Euclidean norm the way np.linalg.norm of a 2-vector evaluates it: sqrt(dx*dx + dy*dy),
    un-fused (the device predicate code is compiled with -fmad=false to round identically)."""
    return np.sqrt(dx * dx + dy * dy)


def nearest_index(p: Sequence[float], ref_xy: np.ndarray) -> int:
    """Global argmin over all reference points, first minimum wins
    (agents/pure_mpc.py:106-109, 566-570, 471-474)."""
    d = _norm2(ref_xy[:, 0] - p[0], ref_xy[:, 1] - p[1])
    return int(np.argmin(d))


# ----------------------------------------------------------------------------------------
# dynamics and cost
# ----------------------------------------------------------------------------------------
def step(s: np.ndarray, u: np.ndarray, dt: float) -> np.ndarray:
    """One explicit-Euler kinematic-bicycle step (agents/pure_mpc.py:220-228, 252-254)."""
    beta = math.atan(REAR_RATIO * math.tan(u[1]))
    return np.array([
        s[0] + dt * s[3] * math.cos(s[2] + beta),
        s[1] + dt * s[3] * math.sin(s[2] + beta),
        s[2] + dt * (s[3] / WHEELBASE) * math.sin(beta),
        s[3] + dt * u[0],
    ])


def rollout(s0: np.ndarray, U: np.ndarray, dt: float = 0.1) -> np.ndarray:
    """X (N+1, 4) from s0 and U (N, 2)."""
    N = U.shape[0]
    X = np.empty((N + 1, 4))
    X[0] = s0
    for k in range(N):
        X[k + 1] = step(X[k], U[k], dt)
    return X


def bound_violation(U: np.ndarray, prob_or_s0, dt: float = 0.1) -> float:
    """Largest violation of the reference's variable bounds (pure_mpc.py:272-280) by the controls U and the
    states they roll out to: |a| <= 5, |delta| <= pi/3, 0 <= v_k <= 30, |theta_k| <= pi for k = 1..N."""
    s0 = getattr(prob_or_s0, "s0", prob_or_s0)
    U = np.asarray(U, dtype=np.float64)
    X = rollout(np.asarray(s0, dtype=np.float64), U, getattr(prob_or_s0, "dt", dt))
    return float(max(0.0, np.abs(U[:, 0]).max() - A_MAX, np.abs(U[:, 1]).max() - DELTA_MAX, V_MIN - X[1:, 3].min(),
                     X[1:, 3].max() - V_MAX, np.abs(X[1:, 2]).max() - TH_MAX))


def repair_feasible(U: np.ndarray, prob_or_s0, dt: float = 0.1) -> np.ndarray:
    """Nearest-in-each-stage feasible controls: walks the horizon and pulls a_k / delta_k back to the edge whenever
    the bound of pure_mpc.py:272-280 on the control itself or on the NEXT node (v_{k+1}, theta_{k+1}; both are
    affine in a_k resp. sin beta(delta_k) under the Euler step of :252-254) would be crossed.  SLSQP returns points
    that violate its inequality constraints by up to its tolerance (and, when it fails, by much more); a yardstick
    cost has to be the cost of a point of the feasible set, so every SLSQP result goes through here first."""
    s0 = np.asarray(getattr(prob_or_s0, "s0", prob_or_s0), dtype=np.float64)
    dt = getattr(prob_or_s0, "dt", dt)
    U = np.array(U, dtype=np.float64)
    s = s0.copy()
    for k in range(U.shape[0]):
        th, v = s[2], s[3]
        a = min(max(U[k, 0], -A_MAX), A_MAX)
        a = min(max(a, (V_MIN - v) / dt), (V_MAX - v) / dt)
        d = min(max(U[k, 1], -DELTA_MAX), DELTA_MAX)
        gain = dt * v / WHEELBASE
        sb = math.sin(math.atan(REAR_RATIO * math.tan(d)))
        if gain > 0.0 and not (TH_MIN <= th + gain * sb <= TH_MAX):
            sb_max = math.sin(math.atan(REAR_RATIO * math.tan(DELTA_MAX)))
            sb = min(max(((TH_MAX if th + gain * sb > TH_MAX else TH_MIN) - th) / gain, -sb_max), sb_max)
            # inverse of sin beta = 0.5 sin d / sqrt(1 - 0.75 sin^2 d)
            d = math.asin(min(max(sb / math.sqrt(0.25 + 0.75 * sb * sb), -1.0), 1.0))
        U[k] = (a, d)
        s = step(s, U[k], dt)
    return U


def step_jacobians(s: np.ndarray, u: np.ndarray, dt: float) -> Tuple[np.ndarray, np.ndarray]:
    """Analytic A = d s+/d s (4x4), B = d s+/d u (4x2) of `step`."""
    t = math.tan(u[1])
    beta = math.atan(REAR_RATIO * t)
    db = REAR_RATIO * (1 + t * t) / (1 + REAR_RATIO * REAR_RATIO * t * t)
    c, sn = math.cos(s[2] + beta), math.sin(s[2] + beta)
    v = s[3]
    A = np.eye(4)
    A[0, 2] = -dt * v * sn
    A[0, 3] = dt * c
    A[1, 2] = dt * v * c
    A[1, 3] = dt * sn
    A[2, 3] = dt * math.sin(beta) / WHEELBASE
    B = np.zeros((4, 2))
    B[0, 1] = -dt * v * sn * db
    B[1, 1] = dt * v * c * db
    B[2, 1] = dt * (v / WHEELBASE) * math.cos(beta) * db
    B[3, 0] = dt
    return A, B


@dataclass
class Problem:
    """One MPC problem after observation parsing / collision logic.

    ref_v[k] is the reference speed seen by stage k (row j(k) = min(ego_index+k, 84) of the
    possibly regenerated table).  `others` rows are (x, y, speed, heading)."""
    s0: np.ndarray
    ego_index: int
    ref_v: np.ndarray                              # (N,)
    N: int = 20
    dt: float = 0.1
    w_speed: float = 1.0                           # already 100 if is_collide (pure_mpc.py:143-147)
    w_control: float = 1.0
    w_input_diff: float = 1.0
    w_distance: float = 0.0                        # 0 = live agent; 10 = archive objective (cfg.yaml:105)
    w_collision: float = 0.0                       # weight on 3000*v^2 term; 0 = live agent
    is_collide: bool = False
    others: np.ndarray = field(default_factory=lambda: np.zeros((0, 4)))
    literal_no_collision: bool = False             # A15: objective = control + input_diff only
    ref_v_final: float = 10.0                      # reference speed at row j(N) (final_state_cost only)

    @property
    def ref(self) -> np.ndarray:
        """The path table of this problem's time step: the reference accumulates its rows with v * dt steps."""
        return path_table(self.dt)


def obstacle_positions(others: np.ndarray, N: int, dt: float) -> np.ndarray:
    """(N, M, 2): position of obstacle i as seen by stage k.  The reference advances the
    deep-copied vehicles by speed*dt*(cos h, sin h) after every stage
    (agents/pure_mpc.py:189-191, agents/base_agent.py:172-174), so stage k sees k steps."""
    M = others.shape[0]
    P = np.empty((N, M, 2))
    pos = others[:, :2].copy()
    inc = others[:, 2:3] * dt * np.stack([np.cos(others[:, 3]), np.sin(others[:, 3])], axis=1) if M else np.zeros((0, 2))
    for k in range(N):
        P[k] = pos
        pos = pos + inc
    return P


def cost_components(X: np.ndarray, U: np.ndarray, prob: Problem) -> np.ndarray:
    """The six un-weighted components [state, control, final_state, input_diff, distance,
    collision] of the reference's `cost_fn` (agents/pure_mpc.py:128-202, 215-216; distance
    term as in agents/archive/pure_mpc.py:189-196; collision term pure_mpc.py:179-183)."""
    N, ref = prob.N, prob.ref
    j = np.minimum(prob.ego_index + np.arange(N), N_REF - 1)
    rx, ry, rh = ref[j, 0], ref[j, 1], ref[j, 3]
    dx, dy = X[:N, 0] - rx, X[:N, 1] - ry
    perp = dx * np.sin(rh) - dy * np.cos(rh)
    para = dx * np.cos(rh) + dy * np.sin(rh)
    state = np.sum(4 * perp**2 + 2 * para**2 + prob.w_speed * (X[:N, 3] - prob.ref_v)**2
                   + 0.5 * (X[:N, 2] - rh)**2)
    control = np.sum(0.01 * U[:, 0]**2 + 0.01 * U[:, 1]**2)
    dU = np.diff(U, axis=0)
    input_diff = np.sum(0.01 * (dU[:, 0]**2 + dU[:, 1]**2))
    J = min(prob.ego_index + N, N_REF - 1)
    final_state = 100 * ((X[N, 0] - ref[J, 0])**2 + (X[N, 1] + ref[J, 1])**2
                         + 20 * (X[N, 3] - prob.ref_v_final)**2 + (X[N, 2] - ref[J, 3])**2)
    distance = 0.0
    if prob.others.shape[0] > 0:
        P = obstacle_positions(prob.others, N, prob.dt)
        d = np.hypot(X[:N, None, 0] - P[:, :, 0], X[:N, None, 1] - P[:, :, 1])
        distance = float(np.sum(np.where(d < 1.0, 1000.0, 100.0) / (d + 1e-6)**2))
    collision = float(np.sum(3000.0 * X[:N, 3]**2)) if prob.is_collide else 0.0
    return np.array([state, control, final_state, input_diff, distance, collision])


def total_cost_from_components(c: np.ndarray, prob: Problem) -> float:
    """agents/pure_mpc.py:204-212 (+ the archive's distance/collision terms when weighted,
    agents/archive/pure_mpc.py:219-226); A15 literal: pure_mpc_no_collision.py:146-151."""
    if prob.literal_no_collision:
        return prob.w_control * c[1] + prob.w_input_diff * c[3]
    return (10.0 * c[0] + prob.w_control * c[1] + prob.w_input_diff * c[3]
            + prob.w_distance * c[4] + prob.w_collision * c[5])


def objective(U: np.ndarray, prob: Problem) -> float:
    X = rollout(prob.s0, U, prob.dt)
    return total_cost_from_components(cost_components(X, U, prob), prob)


def objective_and_sens(Uflat: np.ndarray, prob: Problem):
    """f, grad f (2N,), X (N+1,4), S (N+1, 4, 2N) with S[k] = d X[k] / d U."""
    N, dt, ref = prob.N, prob.dt, prob.ref
    U = Uflat.reshape(N, 2)
    X = np.empty((N + 1, 4))
    S = np.zeros((N + 1, 4, 2 * N))
    X[0] = prob.s0
    for k in range(N):
        A, B = step_jacobians(X[k], U[k], dt)
        X[k + 1] = step(X[k], U[k], dt)
        S[k + 1] = A @ S[k]
        S[k + 1][:, 2 * k:2 * k + 2] += B
    c = cost_components(X, U, prob)
    f = total_cost_from_components(c, prob)
    g = np.zeros(2 * N)
    # control + input-difference parts
    gu = prob.w_control * 0.02 * U
    dU = np.diff(U, axis=0)
    gu[1:] += prob.w_input_diff * 0.02 * dU
    gu[:-1] -= prob.w_input_diff * 0.02 * dU
    g += gu.reshape(-1)
    if not prob.literal_no_collision:
        j = np.minimum(prob.ego_index + np.arange(N), N_REF - 1)
        rx, ry, rh = ref[j, 0], ref[j, 1], ref[j, 3]
        sh, ch = np.sin(rh), np.cos(rh)
        dx, dy = X[:N, 0] - rx, X[:N, 1] - ry
        perp = dx * sh - dy * ch
        para = dx * ch + dy * sh
        lx = np.zeros((N, 4))
        lx[:, 0] = 10 * (8 * perp * sh + 4 * para * ch)
        lx[:, 1] = 10 * (-8 * perp * ch + 4 * para * sh)
        lx[:, 2] = 10 * (X[:N, 2] - rh)
        lx[:, 3] = 10 * 2 * prob.w_speed * (X[:N, 3] - prob.ref_v)
        if prob.w_distance != 0.0 and prob.others.shape[0] > 0:
            P = obstacle_positions(prob.others, N, dt)
            ex, ey = X[:N, None, 0] - P[:, :, 0], X[:N, None, 1] - P[:, :, 1]
            d = np.hypot(ex, ey)
            cc = np.where(d < 1.0, 1000.0, 100.0)
            coef = prob.w_distance * (-2.0 * cc / (d + 1e-6)**3) / np.maximum(d, 1e-300)
            lx[:, 0] += np.sum(coef * ex, axis=1)
            lx[:, 1] += np.sum(coef * ey, axis=1)
        if prob.w_collision != 0.0 and prob.is_collide:
            lx[:, 3] += prob.w_collision * 6000.0 * X[:N, 3]
        g += np.einsum('ki,kij->j', lx, S[:N])
    return f, g, X, S


# ----------------------------------------------------------------------------------------
# NLP solve (single shooting, SLSQP) -- stands in for CasADi/IPOPT, pure_mpc.py:230-318
# ----------------------------------------------------------------------------------------
@dataclass
class Solution:
    U: np.ndarray
    X: np.ndarray
    cost: float
    components: np.ndarray
    success: bool
    nit: int
    message: str = ""

    @property
    def u0(self) -> np.ndarray:
        return self.U[0].copy()


def solve_nlp(prob: Problem, U0: Optional[np.ndarray] = None, ftol: float = 1e-14,
              maxiter: int = 600, enforce_xy: bool = False) -> Solution:
    """Minimise the objective over U with the reference's simple bounds on u
    (pure_mpc.py:278-280) and the state bounds of pure_mpc.py:272-274 applied to stages
    1..N as inequality constraints (stage 0 is fixed by the initial-condition equality).
    Cold start U = 0 as pure_mpc.py:244.  |x|,|y| <= 500 is checked afterwards unless
    `enforce_xy` (never active on this 100 m map)."""
    from scipy.optimize import minimize

    N = prob.N
    cache = {}

    def ev(u):
        key = u.tobytes()
        if key not in cache:
            cache.clear()
            cache[key] = objective_and_sens(u, prob)
        return cache[key]

    def fun(u):
        return ev(u)[0]

    def jac(u):
        return ev(u)[1]

    def cons(u):
        X = ev(u)[2]
        v, th = X[1:, 3], X[1:, 2]
        parts = [v - V_MIN, V_MAX - v, th - TH_MIN, TH_MAX - th]
        if enforce_xy:
            parts += [XY_MAX - X[1:, 0], XY_MAX + X[1:, 0], XY_MAX - X[1:, 1], XY_MAX + X[1:, 1]]
        return np.concatenate(parts)

    def cons_jac(u):
        S = ev(u)[3]
        Sv, Sth = S[1:, 3, :], S[1:, 2, :]
        parts = [Sv, -Sv, Sth, -Sth]
        if enforce_xy:
            parts += [-S[1:, 0, :], S[1:, 0, :], -S[1:, 1, :], S[1:, 1, :]]
        return np.concatenate(parts, axis=0)

    u_init = np.zeros(2 * N) if U0 is None else np.asarray(U0, dtype=np.float64).reshape(-1)
    bounds = [(-A_MAX, A_MAX), (-DELTA_MAX, DELTA_MAX)] * N
    res = minimize(fun, u_init, jac=jac, bounds=bounds, method="SLSQP",
                   constraints=[{"type": "ineq", "fun": cons, "jac": cons_jac}],
                   options={"ftol": ftol, "maxiter": maxiter})
    U = np.clip(res.x.reshape(N, 2), [-A_MAX, -DELTA_MAX], [A_MAX, DELTA_MAX])
    X = rollout(prob.s0, U, prob.dt)
    comp = cost_components(X, U, prob)
    return Solution(U=U, X=X, cost=total_cost_from_components(comp, prob), components=comp,
                    success=bool(res.success), nit=int(res.nit), message=str(res.message))


def kkt_residual(U: np.ndarray, prob: Problem, act_tol: float = 1e-6) -> Tuple[float, float]:
    """Solver-independent optimality certificate.  Returns (stationarity residual,
    max bound violation): with the constraints that are within `act_tol` of active, find
    multipliers mu >= 0 minimising ||grad f - J_act^T mu|| (NNLS)."""
    from scipy.optimize import nnls

    N = prob.N
    f, g, X, S = objective_and_sens(np.asarray(U, dtype=np.float64).reshape(-1), prob)
    rows = []
    viol = 0.0
    Uf = np.asarray(U).reshape(-1)
    lo = np.tile([-A_MAX, -DELTA_MAX], N)
    hi = np.tile([A_MAX, DELTA_MAX], N)
    viol = max(viol, float(np.max(lo - Uf)), float(np.max(Uf - hi)))
    for i in range(2 * N):
        e = np.zeros(2 * N)
        e[i] = 1.0
        if Uf[i] - lo[i] <= act_tol:
            rows.append(e)            # constraint u_i - lo >= 0, gradient +e
        if hi[i] - Uf[i] <= act_tol:
            rows.append(-e)
    for k in range(1, N + 1):
        for idx, (lb, ub) in ((3, (V_MIN, V_MAX)), (2, (TH_MIN, TH_MAX))):
            val = X[k, idx]
            viol = max(viol, lb - val, val - ub)
            if val - lb <= act_tol:
                rows.append(S[k, idx, :])
            if ub - val <= act_tol:
                rows.append(-S[k, idx, :])
    if rows:
        Jt = np.array(rows).T
        mu, rn = nnls(Jt, g)
        return float(rn), float(max(viol, 0.0))
    return float(np.linalg.norm(g)), float(max(viol, 0.0))


def solve_nlp_multiple_shooting(prob: Problem, maxiter: int = 800, ftol: float = 1e-14) -> Solution:
    """Literal restatement of the reference's NLP (agents/pure_mpc.py:230-300):
    z = [vec(X) (4(N+1)), vec(U) (2N)], equality constraints x_0 = s0 and the Euler
    steps, simple bounds on every variable, initial guess = states tiled at s0 and zero
    controls.  Slow (SLSQP on 6N+4 variables); used only for cross-checks."""
    from scipy.optimize import minimize

    N, dt = prob.N, prob.dt
    nx = 4 * (N + 1)

    def unpack(z):
        return z[:nx].reshape(N + 1, 4), z[nx:].reshape(N, 2)

    def fun(z):
        X, U = unpack(z)
        return total_cost_from_components(cost_components(X, U, prob), prob)

    def jac(z):
        X, U = unpack(z)
        # gradient of the separable objective wrt X and U: reuse the single-shooting stage
        # derivative code by finite structure (explicit formulas)
        g = np.zeros_like(z)
        gX = g[:nx].reshape(N + 1, 4)
        gU = g[nx:].reshape(N, 2)
        gU += prob.w_control * 0.02 * U
        dU = np.diff(U, axis=0)
        gU[1:] += prob.w_input_diff * 0.02 * dU
        gU[:-1] -= prob.w_input_diff * 0.02 * dU
        if not prob.literal_no_collision:
            j = np.minimum(prob.ego_index + np.arange(N), N_REF - 1)
            ref = prob.ref
            rx, ry, rh = ref[j, 0], ref[j, 1], ref[j, 3]
            sh, ch = np.sin(rh), np.cos(rh)
            dx, dy = X[:N, 0] - rx, X[:N, 1] - ry
            perp = dx * sh - dy * ch
            para = dx * ch + dy * sh
            gX[:N, 0] = 10 * (8 * perp * sh + 4 * para * ch)
            gX[:N, 1] = 10 * (-8 * perp * ch + 4 * para * sh)
            gX[:N, 2] = 10 * (X[:N, 2] - rh)
            gX[:N, 3] = 20 * prob.w_speed * (X[:N, 3] - prob.ref_v)
            if prob.w_distance != 0.0 and prob.others.shape[0] > 0:
                P = obstacle_positions(prob.others, N, dt)
                ex, ey = X[:N, None, 0] - P[:, :, 0], X[:N, None, 1] - P[:, :, 1]
                d = np.hypot(ex, ey)
                cc = np.where(d < 1.0, 1000.0, 100.0)
                coef = prob.w_distance * (-2.0 * cc / (d + 1e-6)**3) / np.maximum(d, 1e-300)
                gX[:N, 0] += np.sum(coef * ex, axis=1)
                gX[:N, 1] += np.sum(coef * ey, axis=1)
            if prob.w_collision != 0.0 and prob.is_collide:
                gX[:N, 3] += prob.w_collision * 6000.0 * X[:N, 3]
        return g

    def eq(z):
        X, U = unpack(z)
        r = np.empty((N + 1, 4))
        r[0] = X[0] - prob.s0
        for k in range(N):
            r[k + 1] = X[k + 1] - step(X[k], U[k], dt)
        return r.reshape(-1)

    def eq_jac(z):
        X, U = unpack(z)
        Jm = np.zeros((nx, z.size))
        Jm[:4, :4] = np.eye(4)
        for k in range(N):
            A, B = step_jacobians(X[k], U[k], dt)
            r0 = 4 * (k + 1)
            Jm[r0:r0 + 4, r0:r0 + 4] = np.eye(4)
            Jm[r0:r0 + 4, 4 * k:4 * k + 4] = -A
            Jm[r0:r0 + 4, nx + 2 * k:nx + 2 * k + 2] = -B
        return Jm

    z0 = np.concatenate([np.tile(prob.s0, N + 1), np.zeros(2 * N)])
    bounds = [(-XY_MAX, XY_MAX), (-XY_MAX, XY_MAX), (TH_MIN, TH_MAX), (V_MIN, V_MAX)] * (N + 1) \
        + [(-A_MAX, A_MAX), (-DELTA_MAX, DELTA_MAX)] * N
    res = minimize(fun, z0, jac=jac, bounds=bounds, method="SLSQP",
                   constraints=[{"type": "eq", "fun": eq, "jac": eq_jac}],
                   options={"ftol": ftol, "maxiter": maxiter})
    X, U = unpack(res.x)
    U = U.copy()
    Xr = rollout(prob.s0, U, dt)
    comp = cost_components(Xr, U, prob)
    return Solution(U=U, X=Xr, cost=total_cost_from_components(comp, prob), components=comp,
                    success=bool(res.success), nit=int(res.nit), message=str(res.message))


# ----------------------------------------------------------------------------------------
# collision prediction (agents/pure_mpc.py:459-676)
# ----------------------------------------------------------------------------------------
def predict_ego_polyline(pos: np.ndarray, speed: float, start_index: int, ref_speed: float,
                         dt: float = 0.1, ref: Optional[np.ndarray] = None) -> np.ndarray:
    """Path-following prediction of the ego (agents/pure_mpc.py:459-527): point 0 is the
    actual position; the speed ramps by 3.5*dt up to `ref_speed` (or snaps down to it);
    the travelled arc length is mapped onto the reference polyline from `start_index`
    by a left searchsorted + linear interpolation; stops once past the path end.  `ref` defaults to the table of dt."""
    ref = path_table(dt) if ref is None else ref
    pts = [np.array(pos, dtype=np.float64)]
    rp = ref[start_index:, :2]
    if rp.shape[0] < 2:
        return np.array(pts)                                    # pure_mpc.py:478-479
    seg = _norm2(np.diff(rp[:, 0]), np.diff(rp[:, 1]))
    cum = np.concatenate([[0.0], np.cumsum(seg)])               # sequential sum, as :481-484
    # np.cumsum accumulates left-to-right exactly like the reference's Python loop.
    cur_v, dist = float(speed), 0.0
    for _ in range(PRED_HORIZON):
        if cur_v < ref_speed:
            cur_v = min(cur_v + MAX_ACCEL_PRED * dt, ref_speed)
        else:
            cur_v = ref_speed
        dist += cur_v * dt
        idx = int(np.searchsorted(cum, dist))
        if idx >= rp.shape[0]:
            break
        if idx == 0:
            nxt = rp[0].copy()
        else:
            d0, d1 = cum[idx - 1], cum[idx]
            alpha = (dist - d0) / (d1 - d0) if d1 != d0 else 1.0
            alpha = min(max(alpha, 0.0), 1.0)
            nxt = rp[idx - 1] + alpha * (rp[idx] - rp[idx - 1])
        pts.append(nxt)
    if len(pts) <= 1:
        # pure_mpc.py:525-526 falls back to 30 copies of the current position (a zero-length
        # LineString).  That polyline cannot cross anything; it is reported as a one-point polyline
        # and handled as "detection aborted, degenerate" by detect_collisions.
        return np.array(pts)
    return np.array(pts)


def predict_other_polyline(p: Sequence[float], speed: float, heading: float, dt: float = 0.1) -> np.ndarray:
    """31 points by repeated addition of speed*dt*(cos h, sin h) (agents/pure_mpc.py:529-550) -- in FLOAT32, as the
    reference computes them: under its pinned numpy 2.1.2 (requirements.txt:1, NEP 50) `position` is a float32 slice of
    the observation, `speed` = np.linalg.norm of a float32 slice and `heading` a float32 scalar, and
    `future_positions[-1] + speed * dt * np.array([np.cos(heading), np.sin(heading)])` stays float32 throughout.  This
    is decisive for same-lane traffic: x = 2.0 + 30 tiny float32 increments stays EXACTLY 2.0 -- the track is collinear
    with the path and the LineString branch of pure_mpc.py:618-622 is taken -- whereas float64 accumulation drifts off
    the line by ~1e-6 m.  (`speed` arrives here as the float64 norm and is rounded once; numpy's float32 norm may
    differ from that by one ulp.)"""
    f = np.float32
    sd = f(speed) * f(dt)
    h = f(heading)
    inc = sd * np.array([np.cos(h), np.sin(h)], dtype=np.float32)
    cur = np.array(p, dtype=np.float32)
    pts = [cur]
    for _ in range(PRED_HORIZON):
        cur = cur + inc
        pts.append(cur)
    return np.array(pts, dtype=np.float64)


def _orient(ax, ay, bx, by, cx, cy):
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax)


def polyline_intersections(E: np.ndarray, O: np.ndarray, degenerate_eps: float = 1e-9):
    """Intersection candidates of two polylines, standing in for
    `LineString(E).intersection(LineString(O))` + the geometry-type dispatch of
    agents/pure_mpc.py:608-633.  E = the ego's polyline, O = the other vehicle's straight 31-point track.

    * Proper crossings and exact endpoint touches of segment pairs yield points (deduplicated), returned in
      lexicographic (x, then y) order -- the order GEOS' overlay emits the members of a MultiPoint, as far as it can be
      established without GEOS (ASSUMPTION, see DESIGN.md).
    * Collinear overlaps (an ego segment and the track on the same line, all four orientations exactly zero -- the
      same-lane case: highway-env's lane centre x = 2.0 is the reference path's own x) make GEOS return a
      LineString per connected overlap whose coordinates are the merged vertices of both inputs inside the overlap;
      the reference takes `coords[len(coords) // 2]` (pure_mpc.py:618-622, :628-633).  Vertex order: along the ego
      polyline, the first operand of `ego_path.intersection(agent_path)` (ASSUMPTION; it only matters for an even
      number of vertices).  Isolated points that lie on an overlap belong to it.
    * A result that mixes overlaps with isolated points is a GeometryCollection, which the reference's dispatch does
      not handle: no candidate at all (pure_mpc.py:615-633 has no branch for it).
    Returns (points (K,2), degenerate flag): the flag is set when a tested orientation is within
    `degenerate_eps` (relative) of zero WITHOUT being exactly zero, i.e. when GEOS' robust predicates and
    plain FP64 could disagree."""
    ne, no = E.shape[0] - 1, O.shape[0] - 1
    if ne < 1 or no < 1:
        return np.zeros((0, 2)), False
    p1, p2 = E[:-1, None, :], E[1:, None, :]
    q1, q2 = O[None, :-1, :], O[None, 1:, :]
    d1 = _orient(q1[..., 0], q1[..., 1], q2[..., 0], q2[..., 1], p1[..., 0], p1[..., 1])
    d2 = _orient(q1[..., 0], q1[..., 1], q2[..., 0], q2[..., 1], p2[..., 0], p2[..., 1])
    d3 = _orient(p1[..., 0], p1[..., 1], p2[..., 0], p2[..., 1], q1[..., 0], q1[..., 1])
    d4 = _orient(p1[..., 0], p1[..., 1], p2[..., 0], p2[..., 1], q2[..., 0], q2[..., 1])
    scale = (np.abs(p2 - p1).sum(-1) + 1e-300) * (np.abs(q2 - q1).sum(-1) + 1e-300) + 1e-300
    proper = (d1 * d2 < 0) & (d3 * d4 < 0)
    pts: List[Tuple[float, float]] = []
    degenerate = False
    ii, jj = np.nonzero(proper)
    for i, j in zip(ii, jj):
        t = d1[i, j] / (d1[i, j] - d2[i, j])
        pts.append((E[i, 0] + t * (E[i + 1, 0] - E[i, 0]), E[i, 1] + t * (E[i + 1, 1] - E[i, 1])))
    bb = ((np.minimum(p1[..., 0], p2[..., 0]) <= np.maximum(q1[..., 0], q2[..., 0]) + 1e-9)
          & (np.minimum(q1[..., 0], q2[..., 0]) <= np.maximum(p1[..., 0], p2[..., 0]) + 1e-9)
          & (np.minimum(p1[..., 1], p2[..., 1]) <= np.maximum(q1[..., 1], q2[..., 1]) + 1e-9)
          & (np.minimum(q1[..., 1], q2[..., 1]) <= np.maximum(p1[..., 1], p2[..., 1]) + 1e-9))
    near = ((np.abs(d1) <= degenerate_eps * scale) | (np.abs(d2) <= degenerate_eps * scale)
            | (np.abs(d3) <= degenerate_eps * scale) | (np.abs(d4) <= degenerate_eps * scale))
    allzero = (d1 == 0) & (d2 == 0) & (d3 == 0) & (d4 == 0)
    # ---- collinear overlaps: the track is one straight line, so "ego segment i lies on it" does not depend on j
    O0, O1 = O[0], O[-1]
    dO = O1 - O0
    ax = 0 if abs(dO[0]) >= abs(dO[1]) else 1          # scalar coordinate along the line: the dominant axis
    olo, ohi = min(O0[ax], O1[ax]), max(O0[ax], O1[ax])
    pieces = []                                         # [lo, hi] along `ax`, in ego order, touching pieces merged
    on_line = np.zeros(ne, bool)
    if ohi > olo:
        for i in range(ne):
            if not np.all(allzero[i]):
                continue
            a, b = E[i][ax], E[i + 1][ax]
            if a == b:
                continue
            on_line[i] = True
            lo, hi = max(min(a, b), olo), min(max(a, b), ohi)
            if hi > lo:
                if pieces and (pieces[-1][0] == hi or pieces[-1][1] == lo):
                    pieces[-1] = [min(pieces[-1][0], lo), max(pieces[-1][1], hi), pieces[-1][2]]
                else:
                    pieces.append([lo, hi, 1 if b > a else -1])
    # ---- touches (exactly zero orientation with the touching endpoint on the other segment) and near-degenerate pairs
    touch = near & bb & ~proper
    if np.any(touch):
        ti, tj = np.nonzero(touch)
        for i, j in zip(ti, tj):
            if on_line[i]:
                continue                                 # handled as an overlap
            a, b, c, d = E[i], E[i + 1], O[j], O[j + 1]
            o = (d1[i, j], d2[i, j], d3[i, j], d4[i, j])

            def on_seg(p, s, e):
                return (min(s[0], e[0]) <= p[0] <= max(s[0], e[0]) and min(s[1], e[1]) <= p[1] <= max(s[1], e[1]))
            exact = [o[0] == 0 and on_seg(a, c, d), o[1] == 0 and on_seg(b, c, d),
                     o[2] == 0 and on_seg(c, a, b), o[3] == 0 and on_seg(d, a, b)]
            for flag, p in zip(exact, (a, b, c, d)):
                if flag:
                    pts.append((float(p[0]), float(p[1])))
            if any(v != 0 and abs(v) <= degenerate_eps * scale[i, j] for v in o):
                degenerate = True                        # near zero but not zero: robust and plain predicates may differ
    if pieces:
        # isolated points that are not part of an overlap -> GeometryCollection -> the reference finds nothing
        def in_piece(p):
            return any(lo <= p[ax] <= hi for lo, hi, _ in pieces) and _orient(O0[0], O0[1], O1[0], O1[1], p[0], p[1]) == 0
        if any(not in_piece(p) for p in pts):
            return np.zeros((0, 2)), degenerate
        mids = []
        for lo, hi, sgn in pieces:
            vs = [tuple(v) for v in E if lo <= v[ax] <= hi and _orient(O0[0], O0[1], O1[0], O1[1], v[0], v[1]) == 0]
            vs += [tuple(v) for v in O if lo <= v[ax] <= hi]
            vs = sorted(vs, key=lambda v: sgn * v[ax])              # stable: ego vertices before track vertices
            vs = [v for k, v in enumerate(vs) if k == 0 or v[ax] != vs[k - 1][ax]]   # one vertex per position on the line
            mids.append(vs[len(vs) // 2])
        return np.array(mids, dtype=np.float64), degenerate
    if not pts:
        return np.zeros((0, 2)), degenerate
    arr = np.unique(np.array(pts), axis=0)      # lexicographic (x, y) + exact dedup
    return arr, degenerate


@dataclass
class CollisionResult:
    agent_collide: List[bool]
    conflict_index: List[Optional[int]]
    conflict_points: List[Optional[np.ndarray]]
    is_collide: bool
    degenerate: bool
    aborted: bool = False


def detect_collisions(ego: np.ndarray, others: np.ndarray, dt: float = 0.1,
                      ref: Optional[np.ndarray] = None) -> CollisionResult:
    """The detection body of `_check_collision` (agents/pure_mpc.py:565-661), without the
    latch.  `ego` = (x, y, theta, v); `others` rows (x, y, speed, heading).  `ref` defaults to the table of dt."""
    ref = path_table(dt) if ref is None else ref
    ref_xy = ref[:, :2]
    ego_index = nearest_index(ego[:2], ref_xy)
    E = predict_ego_polyline(ego[:2], ego[3], ego_index, ref[ego_index, 2], dt, ref)
    if E.shape[0] < 2:
        # LineString() of one point raises GEOSException -> early return, state left stale
        return CollisionResult([], [], [], False, True, aborted=True)
    flags, idxs, cpts = [], [], []
    degenerate = False
    for o in others:
        O = predict_other_polyline(o[:2], o[2], o[3], dt)
        cand, deg = polyline_intersections(E, O)
        degenerate |= deg
        hit, cidx, cpt = False, None, None
        for q in cand:
            te = int(np.argmin(_norm2(E[:, 0] - q[0], E[:, 1] - q[1])))
            to = int(np.argmin(_norm2(O[:, 0] - q[0], O[:, 1] - q[1])))
            if abs(te - to) < TIME_THRESHOLD:
                hit, cidx, cpt = True, nearest_index(q, ref_xy), np.array(q)
                break
        flags.append(hit)
        idxs.append(cidx)
        cpts.append(cpt)
    return CollisionResult(flags, idxs, cpts, bool(any(flags)), degenerate)


def regenerate_ref_speed(ego_index: int, v_ego: float, is_collide: bool,
                         conflict_index: Sequence[Optional[int]],
                         ref_speed_override: Optional[float] = None,
                         ref: Optional[np.ndarray] = None) -> Tuple[np.ndarray, Optional[int]]:
    """Speed column of `update_reference_states` (agents/pure_mpc.py:678-724).
    Returns (ref_speed[85], stop_index or None).  Only the speed column of `ref` is read (10 at every dt)."""
    ref = path_table() if ref is None else ref
    col = ref[:, 2].copy()
    if ref_speed_override is not None:                         # :683-688, takes precedence
        col[:] = min(max(float(ref_speed_override), 0.0), 30.0)
        return col, None
    if not is_collide:
        return col, None
    valid = [i for i in conflict_index if i is not None]
    if not valid:
        return col, None
    stop = max(ego_index + 1, min(valid) - SAFETY_BUFFER_POINTS)
    stop = min(stop, N_REF - 1)
    n = stop - ego_index
    if n > 0:
        col[ego_index:stop] = np.linspace(v_ego, 0, n)
        col[stop:] = 0.0
        return col, stop
    return col, None


# ----------------------------------------------------------------------------------------
# agent-level restatement (PureMPC_Agent.predict, agents/pure_mpc.py:68-78)
# ----------------------------------------------------------------------------------------
class OraclePureMPCAgent:
    """Stateful single-problem agent with the reference's predict() contract, including
    the 10-step collision latch (agents/pure_mpc.py:38-43, 552-563, 660-676)."""

    def __init__(self, horizon: int = 20, dt: float = 0.1, vehicles_count: int = 9,
                 weight_speed: float = 1.0, weight_control: float = 1.0,
                 weight_input_diff: float = 1.0, weight_distance: float = 0.0,
                 weight_collision: float = 0.0, collision_check: bool = True,
                 literal_no_collision: bool = False):
        self.N, self.dt, self.vehicles_count = horizon, dt, vehicles_count
        self.default_weights = (weight_speed, weight_control, weight_input_diff)
        self.w_distance, self.w_collision = weight_distance, weight_collision
        self.collision_check = collision_check
        self.literal_no_collision = literal_no_collision
        self.ref = path_table(dt)
        self.collision_memory = 0
        self.memorized_conflict_indices: Optional[list] = None
        self.conflict_index: list = []
        self.is_collide = False
        self.ego_index = 0
        self.last_solution: Optional[Solution] = None
        self.last_problem: Optional[Problem] = None

    def check_collision(self, parsed: ParsedObs) -> None:
        if self.collision_memory > 0 and self.memorized_conflict_indices is not None:
            self.conflict_index = self.memorized_conflict_indices
            self.is_collide = True
            self.collision_memory -= 1
            return
        res = detect_collisions(parsed.ego, parsed.others, self.dt, self.ref)
        if res.aborted:
            return
        self.conflict_index = res.conflict_index
        self.is_collide = res.is_collide
        if self.is_collide:
            self.collision_memory = MEMORY_STEPS
            self.memorized_conflict_indices = list(res.conflict_index)
        elif self.collision_memory > 0:
            self.collision_memory -= 1
            self.is_collide = True
        else:
            self.memorized_conflict_indices = None

    def build_problem(self, parsed: ParsedObs, weights_from_RL=None, ref_speed=None) -> Problem:
        w = self.default_weights if weights_from_RL is None else tuple(float(x) for x in np.asarray(weights_from_RL)[0, :3])
        self.ego_index = nearest_index(parsed.ego[:2], self.ref[:, :2])
        override = None if ref_speed is None else float(np.asarray(ref_speed)[0, 0])
        conflict = self.conflict_index
        if self.collision_memory > 0 and self.memorized_conflict_indices is not None:
            conflict = self.memorized_conflict_indices
        col, _ = regenerate_ref_speed(self.ego_index, parsed.ego[3], self.is_collide, conflict, override, self.ref)
        j = np.minimum(self.ego_index + np.arange(self.N), N_REF - 1)
        return Problem(s0=parsed.ego.copy(), ego_index=self.ego_index, ref_v=col[j], N=self.N, dt=self.dt,
                       w_speed=COLLIDE_SPEED_WEIGHT if self.is_collide else w[0],
                       w_control=w[1], w_input_diff=w[2], w_distance=self.w_distance,
                       w_collision=self.w_collision, is_collide=bool(self.is_collide),
                       others=parsed.others.copy(), literal_no_collision=self.literal_no_collision,
                       ref_v_final=float(col[min(self.ego_index + self.N, N_REF - 1)]))

    def predict(self, obs: np.ndarray, return_numpy: bool = True, weights_from_RL=None, ref_speed=None):
        parsed = parse_obs(obs, self.vehicles_count)
        if self.collision_check:
            self.check_collision(parsed)
        prob = self.build_problem(parsed, weights_from_RL, ref_speed)
        sol = solve_nlp(prob)
        self.last_problem, self.last_solution = prob, sol
        return sol.u0
