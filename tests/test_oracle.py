"""The oracle against everything that can pin it without the reference's third-party solver:
the reference's own path table (SURVEY section 4 known answers), the optima derived independently
during the survey (appendix A.7), a solver-independent KKT certificate, the literal
multiple-shooting form of agents/pure_mpc.py:230-300, hand-built collision geometry, and the
committed golden fixtures (regression pin of the oracle itself)."""
import numpy as np
import pytest

import helpers
from helpers import orc


def test_reference_path_known_answers_and_the_library_generator(hostsim):
    r = orc.reference_states()
    assert r.shape == (85, 4)
    assert np.allclose(r[0], (2, 49, 10, -np.pi / 2))
    assert np.allclose(r[39], (2, 10, 10, -np.pi / 2))
    assert np.allclose(r[59], (-11.22584979, -2.22584979, 10, -np.pi), atol=1e-8)
    assert np.allclose(r[84], (-36.22584979, -2.22584979, 10, -np.pi), atol=1e-8)
    # the product's python table and the library's C++ generator (csrc/ref_path.h) are bit-identical to the oracle's
    import mpc_rl_for_avs_b200 as pkg
    assert np.array_equal(pkg.reference_path(), r)
    assert np.array_equal(helpers.hostsim_reference_path(hostsim, 0.1), r)


def _mk(s0, **kw):
    ref = helpers.REF
    s0 = np.array(s0, float)
    idx = orc.nearest_index(s0[:2], ref[:, :2])
    return orc.Problem(s0=s0, ego_index=idx, ref_v=ref[np.minimum(idx + np.arange(20), 84), 2].copy(), **kw)


@pytest.mark.parametrize("s0,f,u0", [
    ((2, 45, -np.pi / 2, 8), 125.78764721, (5.0, 0.0)),
    ((3, 30, -np.pi / 2 + 0.1, 5), 3143.38671483, (5.0, -0.62521401)),
    ((-20, -2.2258, -3.13, 9), None, (5.0, -0.06434809)),       # theta >= -pi active
])
def test_survey_optima(s0, f, u0):
    p = _mk(s0)
    s = orc.solve_nlp(p)
    assert np.max(np.abs(s.u0 - np.array(u0))) < 1e-5
    if f is not None:
        assert abs(s.cost - f) < 1e-6 * f
    kkt, viol = orc.kkt_residual(s.U, p)
    assert kkt < 1e-5 * (1 + s.cost) and viol < 1e-6


def test_multiple_shooting_form_agrees():
    """The reference's own NLP layout (states and controls as variables, dynamics as equalities,
    pure_mpc.py:230-300) has the same optimum as the single-shooting form the oracle solves."""
    p = _mk((3, 30, -np.pi / 2 + 0.1, 5))
    a, b = orc.solve_nlp(p), orc.solve_nlp_multiple_shooting(p)
    assert np.max(np.abs(a.u0 - b.u0)) < 1e-5 and abs(a.cost - b.cost) < 1e-6 * a.cost


def test_multiple_shooting_form_agrees_on_golden_sample():
    """Same cross-check on fixture problems (incl. RL speed overrides): the reference's own NLP layout and the
    single-shooting form reach the same optimum (cost to 1e-6 relative, first control to 1e-4)."""
    g = helpers.load_golden("golden_track")
    probs, _ = helpers.problems_from_obs(g["obs"][:40], g["ref_speed"][:40], g["has_ref_speed"][:40])
    same = n = 0
    for i in range(0, 40, 5):
        a, b = orc.solve_nlp(probs[i]), orc.solve_nlp_multiple_shooting(probs[i])
        n += 1          # (SLSQP's success flag is not used: on the 124-variable form it often stops on its precision test)
        rel = abs(a.cost - b.cost) / max(1.0, abs(a.cost))
        same += rel < 1e-6 and np.max(np.abs(a.u0 - b.u0)) < 1e-4
    assert same >= n - 1, (n, same)


def test_gradient_matches_finite_differences():
    rng = np.random.default_rng(0)
    others = np.array([[6.0, 40.0, 8.0, -np.pi / 2], [-3.0, 33.0, 7.0, 0.0]])
    p = _mk((2.3, 41, -1.5, 7), w_distance=10.0, others=others, w_collision=1.0, is_collide=True, w_speed=100.0)
    U = rng.normal(size=(20, 2)) * [2, 0.2]
    f, g, _, _ = orc.objective_and_sens(U.reshape(-1), p)
    for i in rng.choice(40, 8, replace=False):
        e = np.zeros(40); e[i] = 1e-6
        fd = (orc.objective((U.reshape(-1) + e).reshape(20, 2), p) - orc.objective((U.reshape(-1) - e).reshape(20, 2), p)) / 2e-6
        assert abs(fd - g[i]) <= 1e-5 * max(1.0, abs(g[i])) + 4e-16 * abs(f) / 1e-6      # + rounding noise of the difference quotient


def test_cost_components_quirks():
    """x_N carries no cost and final_state (with the reference's (y + y_ref) sign) is reported only."""
    p = _mk((2, 45, -np.pi / 2, 8))
    U = np.zeros((20, 2))
    X = orc.rollout(p.s0, U)
    c = orc.cost_components(X, U, p)
    X2 = X.copy(); X2[20] += 5.0
    c2 = orc.cost_components(X2, U, p)
    assert c2[0] == c[0] and c2[2] != c[2]
    assert orc.total_cost_from_components(c, p) == orc.total_cost_from_components(c2, p) == 10 * c[0]
    J = min(p.ego_index + 20, 84)
    ref = helpers.REF
    exp = 100 * ((X[20, 0] - ref[J, 0])**2 + (X[20, 1] + ref[J, 1])**2 + 20 * (X[20, 3] - 10)**2 + (X[20, 2] - ref[J, 3])**2)
    assert abs(c[2] - exp) < 1e-9 * exp
    # A15 literal objective: control + input difference only (pure_mpc_no_collision.py:146-151)
    p.literal_no_collision = True
    assert orc.solve_nlp(p).cost < 1e-12


def test_collision_geometry_and_regeneration():
    ref = helpers.REF
    ego = np.array([2.0, 40.0, -np.pi / 2, 10.0])                      # on the path, row 9
    crossing = np.array([[-10.3, 25.4, 8.0, 0.0]])                      # drives +x through (2, 25.4)
    res = orc.detect_collisions(ego, crossing)
    assert res.agent_collide == [True] and not res.degenerate
    assert res.conflict_index[0] == orc.nearest_index((2.0, 25.4), ref[:, :2]) == 24
    assert np.allclose(res.conflict_points[0], (2.0, 25.4))
    # a crossing exactly through an ego polyline vertex (orientation exactly zero) is a genuine point, not degenerate
    res = orc.detect_collisions(ego, np.array([[-10.0, 25.0, 8.0, 0.0]]))
    assert res.agent_collide == [True] and not res.degenerate and np.allclose(res.conflict_points[0], (2.0, 25.0))
    # ... a hair off the vertex is: robust and plain predicates could differ
    Ee = orc.predict_ego_polyline(ego[:2], 10.0, 9, 10.0)
    Oo = orc.predict_other_polyline((-10.0, 25.0), 8.0, 0.0) + (0.0, 2e-10)
    assert orc.polyline_intersections(Ee, Oo)[1]
    # same lane (agents/pure_mpc.py:618-622): a vehicle exactly on the lane centre x = 2.0 heading -pi/2 -- its float32
    # track stays on the path's line, GEOS returns the overlap as a LineString and the reference takes coords[len // 2]
    lead = np.array([[2.0, 30.0, 5.0, float(np.float32(-np.pi / 2))]])
    res = orc.detect_collisions(np.array([2.03, 45.0, -np.pi / 2, 8.0]), lead)
    O = orc.predict_other_polyline(lead[0, :2], 5.0, lead[0, 3])
    assert np.all(O[:, 0] == 2.0) and abs(O[-1, 1] - 15.0) < 1e-4            # exactly on the line, 30 x 0.5 m down
    assert res.agent_collide == [True] and not res.degenerate
    E = orc.predict_ego_polyline((2.03, 45.0), 8.0, orc.nearest_index((2.03, 45.0), ref[:, :2]), 10.0)
    lo, hi = max(E[-1, 1], O[-1, 1]), min(E[1, 1], O[0, 1])                  # overlap of the two spans on x = 2
    merged = sorted({y for y in E[1:, 1] if lo <= y <= hi} | {y for y in O[:, 1] if lo <= y <= hi}, reverse=True)
    assert res.conflict_points[0][0] == 2.0 and res.conflict_points[0][1] == merged[len(merged) // 2]
    # behind the ego: the overlap is empty, nothing is flagged
    assert orc.detect_collisions(np.array([2.03, 45.0, -np.pi / 2, 8.0]), np.array([[2.0, 70.0, 5.0, lead[0, 3]]])).agent_collide == [False]
    # an overlap plus an isolated crossing would be a GeometryCollection, which pure_mpc.py:615-633 does not dispatch on
    O2 = np.array([[1.0, 0.0], [2.0, 0.0], [3.0, 0.0]])
    E2 = np.array([[0.0, 0.0], [1.5, 0.0], [1.5, 4.0], [2.5, 4.0], [2.5, -4.0]])
    pts, deg = orc.polyline_intersections(E2, O2)
    assert len(pts) == 0 and not deg
    # ... while a crossing ON the overlap belongs to it: LineString, middle of the merged vertices (1, 2, 3, 4 -> index 2)
    E3 = np.array([[0.0, 0.0], [4.0, 0.0], [4.0, 4.0], [2.0, 4.0], [2.0, -4.0]])
    pts, deg = orc.polyline_intersections(E3, O2)
    assert pts.tolist() == [[2.0, 0.0]] and not deg
    away = np.array([[10.0, 25.4, 8.0, 0.0]])                           # same lane, already past x = 2
    assert orc.detect_collisions(ego, away).agent_collide == [False]
    parallel = np.array([[-2.0, 0.0, 8.0, np.pi / 2]])                  # opposite lane, never crosses within 3 s
    assert orc.detect_collisions(ego, parallel).is_collide is False
    # regeneration (pure_mpc.py:707-716): stop = max(idx + 1, conflict - 5), linspace(v, 0, n), zeros after
    col, stop = orc.regenerate_ref_speed(9, 10.0, True, [24])
    assert stop == 19 and np.allclose(col[9:19], np.linspace(10, 0, 10)) and np.all(col[19:] == 0) and np.all(col[:9] == 10)
    # RL override takes precedence and is clipped to [0, 30]
    col, stop = orc.regenerate_ref_speed(9, 10.0, True, [24], ref_speed_override=45.0)
    assert stop is None and np.all(col == 30.0)
    # conflict right ahead: stop row is at least idx + 1 -> one ramp point [v]
    col, stop = orc.regenerate_ref_speed(9, 7.0, True, [10])
    assert stop == 10 and col[9] == 7.0 and np.all(col[10:] == 0)


def test_latch_state_machine():
    """One detection, ten latched calls, then detection again (SURVEY A.4)."""
    import mpc_rl_for_avs_b200 as pkg
    obs = np.zeros((3, 8), np.float32)
    obs[0] = (1, 2.0, 40.0, 0.0, -10.0, -np.pi / 2, -1.0, 0.0)
    obs[1] = (1, -10.0, 25.0, 8.0, 0.0, 0.0, 0.0, 1.0)
    ag = orc.OraclePureMPCAgent(horizon=20, vehicles_count=3)
    mems, flags = [], []
    clear = obs.copy(); clear[1, 0] = 0.0                                # the other vehicle disappears
    for step in range(13):
        ag.check_collision(orc.parse_obs(obs if step == 0 else clear, 3))
        mems.append(ag.collision_memory); flags.append(bool(ag.is_collide))
    assert mems == [10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0, 0, 0]
    assert flags == [True] * 11 + [False, False]
    assert pkg is not None


def test_oracle_reproduces_golden_fixtures():
    """Regression pin of the oracle: a sample of each committed fixture is re-derived."""
    for name in ("golden_track", "golden_coll"):
        g = helpers.load_golden(name)
        probs, _ = helpers.problems_from_obs(g["obs"][:24], g["ref_speed"][:24], g["has_ref_speed"][:24],
                                             w_distance=float(g["w_distance"]), collision_check=bool(g["collision_check"]))
        d = helpers.batch_from_problems(probs, int(g["n_obstacles"]))
        for k, v in d.items():
            assert np.array_equal(v, g["batch_" + k][..., :24] if v.ndim > 1 else g["batch_" + k][:24]), k
        import ipm_oracle as ipm
        for i in (0, 12):
            b = ipm.best_known_optimum(probs[i])
            assert abs(b["cost"] - g["oracle_cost"][i]) <= 1e-9 * max(1.0, abs(b["cost"]))
            assert np.allclose(b["U"], g["oracle_U"][i], atol=1e-9) and b["source"] == str(g["oracle_source"][i])
            assert np.allclose(b["ipm_raw_U"], g["ipm_raw_U"][i], atol=1e-9) and b["ipm_status"] == str(g["ipm_status"][i])
            c = orc.cost_components(orc.rollout(probs[i].s0, g["oracle_U"][i]), g["oracle_U"][i], probs[i])
            assert np.allclose(c, g["oracle_components"][i], rtol=1e-9, atol=1e-9)


def test_ipm_oracle_derivatives_and_known_answers():
    """The IPOPT-like interior point on the literal multiple-shooting NLP (oracle/ipm_oracle.py): analytic gradient,
    Jacobian and Lagrangian Hessian against central differences, and the survey's independently derived optima
    (SURVEY A.7) from the reference's own cold start z0 = [tile(s0), 0]."""
    import ipm_oracle as ipm
    ref = helpers.REF
    rng = np.random.default_rng(0)
    s0 = np.array([3, 30, -np.pi / 2 + 0.1, 5.0])
    idx = orc.nearest_index(s0[:2], ref[:, :2])
    others = np.array([[5., 25., 8., np.pi], [0., 20., 7., 0.3]])
    p = orc.Problem(s0=s0, ego_index=idx, ref_v=ref[np.minimum(idx + np.arange(20), 84), 2].copy(), w_distance=10.0, others=others)
    nlp = ipm.LiteralNLP(p)
    assert nlp.n == 124 and nlp.m == 84                                   # agents/pure_mpc.py:260, :249-257
    z = nlp.z0 + rng.normal(0, 0.3, nlp.n)
    g, _ = nlp.grad_hess_f(z, False)
    eps = 1e-6
    E = np.eye(nlp.n)
    gfd = np.array([(nlp.f(z + eps * e) - nlp.f(z - eps * e)) / (2 * eps) for e in E])
    assert np.max(np.abs(g - gfd)) <= 1e-6 * np.max(np.abs(g))
    Jfd = np.array([(nlp.g(z + eps * e) - nlp.g(z - eps * e)) / (2 * eps) for e in E]).T
    assert np.max(np.abs(nlp.jac(z) - Jfd)) <= 1e-7
    lam = rng.normal(0, 1, nlp.m)
    gl = lambda zz: 0.7 * nlp.grad_hess_f(zz, False)[0] + nlp.jac(zz).T @ lam  # noqa: E731
    Hfd = np.array([(gl(z + eps * e) - gl(z - eps * e)) / (2 * eps) for e in E]).T
    H = nlp.hess_lag(z, lam, 0.7)
    assert np.max(np.abs(H - Hfd)) <= 1e-6 * np.max(np.abs(H))
    cases = [((2, 45, -np.pi / 2, 8), 125.78764721, (5.0, 0.0)),
             ((3, 30, -np.pi / 2 + 0.1, 5), 3143.38671483, (5.0, -0.62521401)),
             ((ref[48, 0] + 0.3, ref[48, 1] - 0.2, ref[48, 3] + 0.05, 9), 31.61840094, (5.0, -0.68614018))]
    for s0, f, u0 in cases:
        s0 = np.array(s0, float)
        idx = orc.nearest_index(s0[:2], ref[:, :2])
        pr = orc.Problem(s0=s0, ego_index=idx, ref_v=ref[np.minimum(idx + np.arange(20), 84), 2].copy())
        r = ipm.solve_ipopt_like(pr)
        assert r.success and not r.restoration and r.constr_viol <= 1e-6
        assert np.max(np.abs(r.u0 - np.array(u0))) <= 1e-5 and abs(r.cost - f) <= 1e-7 * f


def test_repair_feasible_projects_onto_the_reference_bounds():
    """mpc_oracle.repair_feasible: identity on feasible controls, exact feasibility (pure_mpc.py:272-280) otherwise, and
    the pulled-back stage sits ON the bound it crossed."""
    rng = np.random.default_rng(5)
    g = helpers.load_golden("golden_holdout")
    probs, _ = helpers.problems_from_obs(g["obs"][:32], g["ref_speed"][:32], g["has_ref_speed"][:32],
                                         w_distance=float(g["w_distance"]), collision_check=True)
    for i, p in enumerate(probs):
        U = g["oracle_U"][i]
        assert orc.bound_violation(U, p) == 0.0                      # the yardstick itself is feasible
        assert np.array_equal(orc.repair_feasible(U, p), U)
        W = np.stack([rng.uniform(-9, 9, p.N), rng.uniform(-1.6, 1.6, p.N)], axis=1)
        R = orc.repair_feasible(W, p)
        assert orc.bound_violation(R, p) <= 1e-12
        X = orc.rollout(p.s0, R, p.dt)
        moved = np.nonzero(np.abs(R - W).max(axis=1) > 0)[0]
        for k in moved:                                              # every change is explained by an active bound
            on_a = abs(abs(R[k, 0]) - 5.0) < 1e-12 or min(abs(X[k + 1, 3]), abs(X[k + 1, 3] - 30.0)) < 1e-9
            on_d = abs(abs(R[k, 1]) - np.pi / 3) < 1e-12 or abs(abs(X[k + 1, 2]) - np.pi) < 1e-9
            assert (R[k, 0] == W[k, 0] or on_a) and (R[k, 1] == W[k, 1] or on_d), (i, k)
    # a braking ramp that would drive the speed negative stops exactly at v = 0
    s0 = np.array([0.0, 0.0, 0.0, 1.0])
    R = orc.repair_feasible(np.tile([-5.0, 0.0], (20, 1)), s0)
    assert np.allclose(orc.rollout(s0, R)[2:, 3], 0.0, atol=1e-15) and np.allclose(R[:2, 0], -5.0) and np.allclose(R[2:, 0], 0.0, atol=1e-12)
