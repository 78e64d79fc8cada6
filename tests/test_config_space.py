"""The CUDA path off the shipped configuration point (dt = 0.1, 8 other vehicles, horizon 20): policy frequencies
1..30 for the path table, the solve at horizons 2..64 with 1..16 other vehicles and at 5 and 20 Hz, the collision
term of the objective, and handles of two frequencies in one process.

The reference builds its 85-row path with v * dt steps (agents/base_agent.py:118-154), so every frequency has its own
table; each handle builds its table from its dt (csrc/ref_path.h) and keeps it in its own device memory."""
import numpy as np
import pytest
import torch

import helpers
from helpers import orc

CFG = {"horizon": 20, "weight_speed": 1.0, "weight_control": 1.0, "weight_input_diff": 1.0}


def test_path_table_generator_matches_oracle_at_every_frequency(hostsim):
    """The library's table generator (what mpc_create uploads) is bit-identical to the oracle's reference_states(1/f) for
    f = 1..30; at f = 10 it is also the table the package's python mirror builds, which the device held before tables
    were built per handle, so default outputs cannot change."""
    for f in range(1, 31):
        dt = 1 / f
        t = helpers.hostsim_reference_path(hostsim, dt)
        assert np.array_equal(t, orc.reference_states(dt)), f
    import mpc_rl_for_avs_b200 as pkg
    assert np.array_equal(helpers.hostsim_reference_path(hostsim, 0.1), pkg.reference_path(0.1))
    # the rows really are dt-dependent: 1 m apart at 10 Hz, 2 m at 5 Hz
    assert orc.reference_states(0.1)[1, 1] - orc.reference_states(0.1)[0, 1] == -1.0
    assert orc.reference_states(0.2)[1, 1] - orc.reference_states(0.2)[0, 1] == -2.0


# (N, M, dt, weight_collision, status-0 bar): a spanning subset of N in {2, 16, 64} x M in {1, 9, 16} at 20 and 5 Hz, and
# the shipped point with the 3000 v^2 collision term weighted.  The bars sit a little below the rates measured on a B200,
# listed in test_solve_off_the_shipped_point's docstring.
SOLVE_CASES = [
    pytest.param(2, 16, 0.2, 0.0, 0.97, id="N2-M16-f5"),
    pytest.param(16, 1, 0.05, 0.0, 0.93, id="N16-M1-f20"),
    pytest.param(16, 9, 0.2, 0.0, 0.9, id="N16-M9-f5"),
    pytest.param(64, 9, 0.05, 0.0, 0.42, id="N64-M9-f20"),
    pytest.param(20, 16, 0.05, 0.0, 0.9, id="N20-M16-f20"),
    pytest.param(20, 8, 0.1, 1.0, 0.88, id="N20-M8-f10-wc1"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,dt,wc,bar", SOLVE_CASES)
def test_solve_off_the_shipped_point(N, M, dt, wc, bar):
    """Every returned iterate satisfies the reference's bounds; the first <= 12 status-0 problems outside degenerate
    scenes are confirmed by the oracle started at them; the status-0 rate meets a bar a little below the measured one.
    Measured status-0 rates on one B200 (1000 W; B = 600, collision logic on, distance weight 10, 4 starts):
    N2-M16-f5 1.000, N16-M1-f20 0.958, N16-M9-f5 0.927, N64-M9-f20 0.463 (most horizons run past the path's end, where
    the NLP is ill-posed), N20-M16-f20 0.932, N20-M8-f10-wc1 0.910.  The start portfolio is tuned at 10 Hz only.  wc1:
    the collision term 3000 v^2 enters the objective of colliding scenes, and its gradient and Hessian only the backward
    sweep."""
    import mpc_rl_for_avs_b200 as pkg
    B = 600
    obs, rs, probs = helpers.config_scenes(B, N, M, dt, seed=100 + N + M)
    for p in probs:
        p.w_collision = wc
    rsn = torch.from_numpy(rs).cuda()
    agent = pkg.BatchedPureMPC(dict(CFG, horizon=N), vehicles_count=M + 1, max_batch=B, dt=dt, collision_check=True,
                               weight_distance=10.0 if M else 0.0, weight_collision=wc, max_iter=80 if N > 40 else 60)
    actions, U = agent.predict_batch(torch.from_numpy(obs).cuda(), ref_speed=rsn, return_controls=True)
    torch.cuda.synchronize()
    U = U.cpu().numpy()
    st = agent.status[:B].cpu().numpy()
    ego = agent.ego_index[:B].cpu().numpy()
    isc = agent.is_collide[:B].cpu().numpy().astype(bool)
    deg = agent.degenerate[:B].cpu().numpy().astype(bool)
    assert np.array_equal(ego, [p.ego_index for p in probs])
    assert np.array_equal(isc[~deg], np.array([p.is_collide for p in probs])[~deg])
    if wc:
        assert isc.mean() >= 0.1
    rate = float((st == 0).mean())
    print(f"N {N} M {M} dt {dt} wc {wc}: status 0 {rate:.3f}, settled {float(((st & ~32) == 0).mean()):.3f}")
    assert rate >= bar, rate
    assert ((st & 4) == 0).all()
    for i in range(B):
        assert np.all(np.abs(U[i][:, 0]) <= 5 + 1e-6) and np.all(np.abs(U[i][:, 1]) <= np.pi / 3 + 1e-6), i
        X = orc.rollout(probs[i].s0, U[i].astype(np.float64), dt)
        assert X[1:, 3].min() >= -1e-4 and X[1:, 3].max() <= 30 + 1e-4 and np.abs(X[1:, 2]).max() <= np.pi + 1e-4, i
    n = 0
    for i in np.nonzero((st == 0) & ~deg)[0][:12]:
        ok, du0, gain = helpers.oracle_warm_confirms(probs[i], U[i], rel_gain_tol=1e-4 if N > 40 else 1e-6)
        assert ok, (i, du0, gain)
        n += 1
    assert n >= 6
    if wc:
        # the weighted collision term is what the returned cost contains
        i = int(np.nonzero((st == 0) & isc & ~deg)[0][0])
        c64 = orc.objective(U[i].astype(np.float64), probs[i])
        assert orc.cost_components(orc.rollout(probs[i].s0, U[i].astype(np.float64), dt), U[i], probs[i])[5] > 0
        near, tol = helpers.distance_conditioning(probs[i], U[i])
        assert near or abs(agent.cost[i].item() - c64) <= 2e-5 * max(1.0, abs(c64)) + 10 * tol


@pytest.mark.gpu
def test_sixteen_vehicles_run_the_192_thread_kernel_and_do_not_depend_on_the_launch():
    """At M = 16 the slot file no longer fits 256 problems per SM: every launch size takes the 192-thread TMEM kernel,
    whose tail compaction is otherwise only reached through a forced block size.  Results for B = 37, 600 and 4096 and
    for a forced 128-thread block (TMEM without compaction) are bit-identical on the shared problems."""
    import mpc_rl_for_avs_b200 as pkg
    M, Bmax = 16, 4096
    obs, rs, has = pkg.make_scenarios(Bmax, M, seed=616)
    rsn = torch.where(has.reshape(-1, 1), rs, torch.full_like(rs, float("nan"))).cuda()
    obs_d = obs.cuda()
    agent = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=Bmax, collision_check=True, weight_distance=10.0)
    ref = None
    for B in (4096, 37, 600):
        sc = agent.solve_config(B)
        assert sc["gains_in_tmem"] and sc["threads_per_block"] == 192, (B, sc)
        agent.reset()
        a = agent.predict_batch(obs_d[:B].contiguous(), ref_speed=rsn[:B].contiguous()).clone()
        st, it = agent.status[:B].clone(), agent.iters[:B].clone()
        if ref is None:
            ref = (a, st, it)
            assert float((st == 0).float().mean()) >= 0.7
            continue
        assert torch.equal(a, ref[0][:B]) and torch.equal(st, ref[1][:B]) and torch.equal(it, ref[2][:B]), B
    forced = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=Bmax, collision_check=True, weight_distance=10.0,
                                threads_per_block=128)
    sc = forced.solve_config(Bmax)
    assert sc["gains_in_tmem"] and sc["threads_per_block"] == 128, sc
    a = forced.predict_batch(obs_d, ref_speed=rsn)
    assert torch.equal(a, ref[0]) and torch.equal(forced.status[:Bmax], ref[1]) and torch.equal(forced.iters[:Bmax], ref[2])


@pytest.mark.gpu
def test_two_policy_frequencies_in_one_process():
    """Handles at dt = 0.1 and dt = 0.2 called alternately on their own scenes: each result is bit-identical to a fresh
    single handle's, and its ego rows and collision flags are those of its own oracle (a table shared by the device
    could serve only one of them)."""
    import mpc_rl_for_avs_b200 as pkg
    B, M = 512, 8
    scenes, fresh = {}, {}
    for dt in (0.1, 0.2):
        obs, _, _ = pkg.make_scenarios(B, M, seed=202, dt=dt, same_lane_frac=0.25)
        scenes[dt] = obs.cuda()
        a = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=B, dt=dt, collision_check=True, weight_distance=10.0)
        fresh[dt] = (a.predict_batch(scenes[dt]).clone(), a.ego_index[:B].clone(), a.agent_collide[:B].clone())
        del a
        torch.cuda.synchronize()
    h = {dt: pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=B, dt=dt, collision_check=True, weight_distance=10.0)
         for dt in (0.1, 0.2)}
    for rnd in range(2):
        for dt in (0.1, 0.2, 0.1, 0.2):
            h[dt].reset()
            a = h[dt].predict_batch(scenes[dt])
            assert torch.equal(a, fresh[dt][0]), (rnd, dt)
            assert torch.equal(h[dt].ego_index[:B], fresh[dt][1]) and torch.equal(h[dt].agent_collide[:B], fresh[dt][2]), (rnd, dt)
    for dt in (0.1, 0.2):
        o = scenes[dt].cpu().numpy()
        ego = fresh[dt][1].cpu().numpy()
        flags = fresh[dt][2].cpu().numpy().astype(bool)
        deg = h[dt].degenerate[:B].cpu().numpy().astype(bool)
        n_deg = 0
        for i in range(B):
            parsed = orc.parse_obs(o[i], M + 1)
            assert ego[i] == orc.nearest_index(parsed.ego[:2], orc.path_table(dt)[:, :2]), (dt, i)
            res = orc.detect_collisions(parsed.ego, parsed.others, dt)
            if res.degenerate or deg[i]:
                n_deg += 1
                continue
            assert list(flags[i]) == list(res.agent_collide), (dt, i)
        assert n_deg <= 0.005 * B
    # the two tables differ where it matters: most scenes of the 5 Hz set have another nearest row on the 10 Hz table
    o = scenes[0.2].cpu().numpy()
    other = [orc.nearest_index(o[i, 0, 1:3].astype(np.float64), orc.path_table(0.1)[:, :2]) for i in range(B)]
    assert np.mean(np.array(other) != fresh[0.2][1].cpu().numpy()) >= 0.9
