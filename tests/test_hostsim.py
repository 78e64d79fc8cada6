"""CPU checks of the SOLVER LOGIC: the kernel's per-problem device functions (mpc_core.cuh) are
compiled for the host by the test-only harness (tests/hostsim) and compared with the oracle, in
float (the device arithmetic) and double.  These mirror the -m gpu parity tests so that the
algorithm is covered where no GPU exists; they do not exercise the CUDA library."""
import numpy as np
import pytest

import helpers
from helpers import orc


def _golden_batch(g):
    return {k[len("batch_"):]: v for k, v in g.items() if k.startswith("batch_")}


def _problems(g):
    probs, _ = helpers.problems_from_obs(g["obs"], g["ref_speed"], g["has_ref_speed"], w_distance=float(g["w_distance"]),
                                         collision_check=bool(g["collision_check"]))
    return probs


def _rollout_inputs(hostsim, name, N, M, wd, dt, B=64):
    """(problems, SoA batch, controls): a golden set, or seeded scenes of the configuration (N, M, dt).  The controls are
    random, and near-optimal for the first quarter (the golden optimum, or the host build's own solution): the cancellation
    regime near an optimum."""
    rng = np.random.default_rng(3)
    U = np.stack([rng.uniform(-5, 5, (B, N)), rng.uniform(-1.0, 1.0, (B, N))], axis=-1).astype(np.float32)
    if name.startswith("golden"):
        g = helpers.load_golden(name)
        probs = _problems(g)[:B]
        d = {k: np.ascontiguousarray(v[..., :B] if v.ndim > 1 else v[:B]) for k, v in _golden_batch(g).items()}
        U[:B // 4] = g["oracle_U"][:B // 4].astype(np.float32)
    else:
        _, _, probs = helpers.config_scenes(B, N, M, dt, seed=11 + N + M)
        d = helpers.batch_from_problems(probs, M)
        r = helpers.hostsim_solve(hostsim, {k: np.ascontiguousarray(v[..., :B // 4]) for k, v in d.items()},
                                  helpers.hs_config(N=N, M=M, dt=dt, w_distance=wd))
        U[:B // 4] = r["U"]
    return probs, d, U


ROLLOUT_CASES = [pytest.param("golden_track", 20, 0, 0.0, 0.1, id="golden_track-0-0.0"),
                 pytest.param("golden_coll", 20, 8, 10.0, 0.1, id="golden_coll-8-10.0")] + [
    pytest.param("scenes", N, M, 10.0 if M else 0.0, dt, id=f"N{N}-M{M}-f{round(1 / dt)}") for N, M, dt in helpers.ROLLOUT_CONFIGS]


@pytest.mark.parametrize("name,N,M,wd,dt", ROLLOUT_CASES)
@pytest.mark.parametrize("use_double", [False, True])
def test_rollout_cost_matches_oracle(hostsim, name, N, M, wd, dt, use_double):
    """Rollout and cost components of the host build against the oracle: the golden sets (H=20, dt=0.1) and the
    configurations of helpers.ROLLOUT_CONFIGS (horizons 2..64, 0..16 other vehicles, policy frequencies 5..20; with
    N >= 16 most horizons run past the path's last row, where the reference row and the final-state row clamp)."""
    probs, d, U = _rollout_inputs(hostsim, name, N, M, wd, dt)
    X, c6, tot = helpers.hostsim_rollout_cost(hostsim, d, helpers.hs_config(N=N, M=M, dt=dt, w_distance=wd), U, use_double)
    if name == "scenes" and N > 20:
        assert sum(p.ego_index + N > 84 for p in probs) >= len(probs) // 8
    helpers.check_rollout_cost(probs, U, X, c6, tot)


@pytest.mark.parametrize("name,M,wd", [("golden_track", 0, 0.0), ("golden_coll", 8, 10.0), ("golden_holdout", 8, 10.0),
                                       ("golden_holdout_1k", 8, 10.0)])
@pytest.mark.parametrize("n_starts", [1, 4])
def test_solver_logic_against_golden(hostsim, name, M, wd, n_starts):
    """Host build of the device code against the best known optimum of the CPU portfolio (IPOPT-like interior point on
    the literal multiple-shooting NLP + SLSQP, oracle/ipm_oracle.py): the bars of helpers.PARITY_BARS."""
    g = helpers.load_golden(name)
    probs = _problems(g)
    B = len(probs)
    r = helpers.hostsim_solve_init(hostsim, _golden_batch(g), helpers.hs_config(M=M, w_distance=wd), n_starts=n_starts)
    st = helpers.solve_parity_stats(r, g, probs)
    helpers.assert_parity_bars(st, name, n_starts)
    # same first control almost always means the same optimum (a shared pinned first control with a
    # different tail is the exception): then the costs agree
    rel = np.abs(st["cost64"] - g["oracle_cost"]) / np.maximum(np.abs(g["oracle_cost"]), 1.0)
    assert np.mean(rel[st["same_mask"] & st["conv_mask"]] <= 1e-4) >= 0.9
    # every converged (status 0) solution is confirmed by the oracle started at it (sample of 32)
    for i in np.nonzero(st["conv_mask"])[0][:32]:
        ok, du0, gain = helpers.oracle_warm_confirms(probs[i], r["U"][i])
        assert ok, (i, du0, gain)
    # every iterate respects the reference's bounds, converged or not
    for i in range(B):
        X = orc.rollout(probs[i].s0, r["U"][i].astype(np.float64))
        assert X[1:, 3].min() >= -1e-4 and X[1:, 3].max() <= 30 + 1e-4 and np.abs(X[1:, 2]).max() <= np.pi + 1e-4


def test_float_and_double_agree_on_converged_problems(hostsim):
    g = helpers.load_golden("golden_track")
    d = _golden_batch(g)
    cfg = helpers.hs_config(M=0)
    rf = helpers.hostsim_solve(hostsim, d, cfg, use_double=False)
    rd = helpers.hostsim_solve(hostsim, d, cfg, use_double=True)
    both = (rf["status"] == 0) & (rd["status"] == 0)
    du = np.max(np.abs(rf["actions"] - rd["actions"]), axis=1)
    assert both.mean() > 0.85
    assert np.mean(du[both] <= 1e-3) >= 0.95      # the rest are different basins reached through rounding


def test_survey_known_answers(hostsim):
    ref = helpers.REF
    cases = [((2, 45, -np.pi / 2, 8), 125.78764721, (5.0, 0.0)),
             ((3, 30, -np.pi / 2 + 0.1, 5), 3143.38671483, (5.0, -0.62521401)),
             ((ref[48, 0] + 0.3, ref[48, 1] - 0.2, ref[48, 3] + 0.05, 9), 31.61840094, (5.0, -0.68614018))]
    probs = []
    for s0, _, _ in cases:
        s0 = np.array(s0, float)
        idx = orc.nearest_index(s0[:2], ref[:, :2])
        probs.append(orc.Problem(s0=s0, ego_index=idx, ref_v=ref[np.minimum(idx + np.arange(20), 84), 2].copy()))
    r = helpers.hostsim_solve(hostsim, helpers.batch_from_problems(probs, 0), helpers.hs_config(M=0))
    for i, (_, f, u0) in enumerate(cases):
        assert np.max(np.abs(r["actions"][i] - np.array(u0))) <= 1e-3
        assert abs(r["cost"][i] - f) <= 1e-4 * f


def test_horizon16_solver_logic(hostsim):
    """Shipped horizon (config/cfg.yaml:90) through the same device functions."""
    import mpc_rl_for_avs_b200 as pkg
    B, M, N = 32, 9, 16
    obs, rs, has = pkg.make_scenarios(B, M, seed=31)
    probs, _ = helpers.problems_from_obs(obs.numpy(), rs.numpy(), has.numpy(), w_distance=10.0, collision_check=True, N=N)
    r = helpers.hostsim_solve(hostsim, helpers.batch_from_problems(probs, M), helpers.hs_config(N=N, M=M, w_distance=10.0))
    conv = r["status"] == 0
    assert conv.mean() >= 0.8
    for i in np.nonzero(conv)[0][:12]:
        ok, du0, gain = helpers.oracle_warm_confirms(probs[i], r["U"][i])
        assert ok, (i, du0, gain)


def test_solver_logic_at_policy_frequency_5(hostsim):
    """dt = 0.2: the problems are built on the path table of that dt (1 m -> 2 m row spacing).  Every status-0 solution
    of a sample of 16 is confirmed by the oracle started at it."""
    B, N, M, dt = 48, 20, 8, 0.2
    _, _, probs = helpers.config_scenes(B, N, M, dt, seed=5)
    r = helpers.hostsim_solve_init(hostsim, helpers.batch_from_problems(probs, M), helpers.hs_config(N=N, M=M, dt=dt, w_distance=10.0),
                                   n_starts=4)
    conv = r["status"] == 0
    assert conv.mean() >= 0.7, conv.mean()
    for i in np.nonzero(conv)[0][:16]:
        ok, du0, gain = helpers.oracle_warm_confirms(probs[i], r["U"][i])
        assert ok, (i, du0, gain)
