"""SURVEY 8-f next rows N1/N2: batched synthetic env + batched A2C-MPC loop.  CPU: env rules and the rollout /
update plumbing with a stub controller; GPU: the real MPC in the loop."""
import math

import numpy as np
import pytest
import torch


class _StubMPC:
    """Constant controller with the BatchedPureMPC.predict_batch signature (CPU plumbing test only)."""

    def predict_batch(self, obs, ref_speed=None, weights=None, reset_mask=None):
        a = torch.zeros(obs.shape[0], 2)
        a[:, 0] = 0.2
        return a


def test_env_rules_cpu():
    from mpc_rl_for_avs_b200.rl import BatchedIntersectionEnv
    env = BatchedIntersectionEnv(16, 9, device="cpu", seed=3)
    obs = env.observe()
    assert obs.shape == (16, 10, 8) and (obs[:, :, 0] == 1).all()
    d = torch.hypot(obs[:, 1:, 1] - obs[:, :1, 1], obs[:, 1:, 2] - obs[:, :1, 2])
    assert (d[:, 1:] >= d[:, :-1]).all()                                   # others sorted by distance (cfg.yaml:4-6)
    assert torch.allclose(obs[:, 0, 5], torch.full((16,), -math.pi / 2))
    # raw SB3 action path (quirk Q8): accel clipped to +-1 then x5
    v0 = env.ego[:, 3].clone()
    obs2, rew, done, info = env.step(torch.tensor([[7.0, 0.0]]).repeat(16, 1))
    assert torch.allclose(env.ego[:, 3][~done], (v0 + 0.5)[~done], atol=1e-5)
    assert ((rew <= 1.0) & (rew >= -5.0)).all()
    # a vehicle parked on the ego's nose crashes it: reward -5, episode ends and the env is reset in place
    env.oth[0, 0, :2] = env.ego[0, :2] + torch.tensor([0.0, -1.0])
    env.oth[0, 0, 2] = 0.0
    _, rew, done, info = env.step(torch.zeros(16, 2))
    assert bool(info["crashed"][0]) and bool(done[0]) and rew[0] <= -4.0 and int(env.t[0]) == 0
    # time limit
    env2 = BatchedIntersectionEnv(4, 9, device="cpu", seed=4, duration_steps=3)
    for _ in range(3):
        _, _, done, info = env2.step(torch.tensor([[-1.0, 0.0]]).repeat(4, 1))
    assert bool((info["truncated"] | info["crashed"]).all())
    # seeded
    a = BatchedIntersectionEnv(8, 9, device="cpu", seed=7).observe()
    b = BatchedIntersectionEnv(8, 9, device="cpu", seed=7).observe()
    assert torch.equal(a, b)


def test_a2c_plumbing_cpu():
    from mpc_rl_for_avs_b200.rl import A2CMPC, BatchedIntersectionEnv
    env = BatchedIntersectionEnv(8, 9, device="cpu", seed=1)
    algo = A2CMPC(env, _StubMPC(), n_steps=5)
    p0 = [p.detach().clone() for p in algo.policy.parameters()]
    log = algo.train_step()
    assert all(np.isfinite(v) for v in log.values())
    assert any(not torch.equal(a, b) for a, b in zip(p0, algo.policy.parameters()))
    assert algo.stats["steps"] == 40


def test_ppo_plumbing_cpu():
    from mpc_rl_for_avs_b200.rl import PPOMPC, BatchedIntersectionEnv
    for version, use_sde in (("v0", True), ("v1", False)):
        env = BatchedIntersectionEnv(8, 9, device="cpu", seed=2, duration_steps=4)     # truncations -> value bootstrap path
        algo = PPOMPC(env, _StubMPC(), n_steps=6, n_epochs=2, batch_size=16, use_sde=use_sde, version=version)
        assert algo.policy.log_std.shape == ((64, algo.action_dim) if use_sde else (algo.action_dim,))
        assert algo.action_dim == (1 if version == "v0" else 3)
        p0 = [p.detach().clone() for p in algo.policy.parameters()]
        log = algo.train_step()
        assert all(np.isfinite(v) for v in log.values()) and "approx_kl" in log
        assert any(not torch.equal(a, b) for a, b in zip(p0, algo.policy.parameters()))
        assert algo.num_timesteps == 48
        # PPO_MPC clips the RL action to the Box before the MPC; A2C_MPC does not (quirk Q6)
        seen = {}

        class Spy(_StubMPC):
            def predict_batch(self, obs, ref_speed=None, weights=None, reset_mask=None):
                seen["rs"], seen["w"] = ref_speed, weights
                return super().predict_batch(obs)
        algo.mpc = Spy()
        algo.mpc_action(env.observe(), torch.full((8, algo.action_dim), 7.0))
        got = seen["rs"] if version == "v0" else seen["w"]
        assert float(got.max()) == 1.0 and got.shape == (8, 1 if version == "v0" else 3)


def test_gsde_likelihood_matches_sampling_cpu():
    """gSDE: noise = latent @ theta, theta ~ N(0, sigma^2) per env; the per-sample std is sqrt(latent^2 @ sigma^2)."""
    from mpc_rl_for_avs_b200.rl import ActorCritic
    torch.manual_seed(0)
    pol = ActorCritic(80, 1, use_sde=True, log_std_init=-1.0)
    obs = torch.randn(1, 80).repeat(20000, 1)
    pol.reset_noise(20000)
    a, _, lp = pol(obs)
    d, _ = pol.dist(obs)
    assert abs(float(a.std()) / float(d.stddev[0]) - 1.0) < 0.03 and abs(float(a.mean() - d.mean[0])) < 0.02
    # same exploration matrix -> same action for the same observation until the next reset_noise
    a2, _, _ = pol(obs)
    assert torch.equal(a, a2)
    v, lp2, ent = pol.evaluate_actions(obs, a)
    assert torch.allclose(lp, lp2)


def test_sb3_zip_checkpoints_cpu(tmp_path):
    from mpc_rl_for_avs_b200 import checkpoint
    from mpc_rl_for_avs_b200.rl import ActorCritic
    torch.manual_seed(1)
    for use_sde in (False, True):
        pol = ActorCritic(80, 1, use_sde=use_sde)
        path = str(tmp_path / f"p{int(use_sde)}.zip")
        checkpoint.save_sb3_policy(path, pol, {"n_steps": 64, "gamma": 0.99})
        pol2, data = checkpoint.load_sb3_policy(path)
        assert pol2.use_sde == use_sde and data["n_steps"] == 64
        x = torch.randn(5, 80)
        assert torch.equal(pol(x, deterministic=True)[0], pol2(x, deterministic=True)[0])
    # checkpoints as Stable-Baselines3 writes the reference's (weights/v0: A2C with a state-independent std, PPO with
    # gSDE): the parameter names and shapes of SB3's MlpPolicy are spelled out below, not taken from ActorCritic, and the
    # loaded policy must compute what that MlpPolicy computes
    rng = np.random.default_rng(5)
    x = rng.standard_normal((5, 10, 8))
    for name, sde, hp in (("test_a2c_v0.zip", False, {"n_steps": 64, "learning_rate": 0.0007, "num_timesteps": 128}),
                          ("test_ppo_v0.zip", True, {"n_steps": 64, "batch_size": 64, "n_epochs": 10, "num_timesteps": 256})):
        sd = _sb3_mlp_policy_state(rng, 80, 1, sde)
        path = str(tmp_path / name)
        _write_sb3_layout_zip(path, sd, sde, hp)
        pol, data = checkpoint.load_sb3_policy(path)
        assert pol.use_sde == sde and data["observation_space_shape"] == (10, 8) and data["action_space_shape"] == (1,)
        assert all(data[k] == v for k, v in hp.items()) and "policy_class" not in data and "lr_schedule" not in data
        a, v, lp = pol(torch.zeros(3, 80), deterministic=True)
        assert a.shape == (3, 1) and torch.isfinite(a).all() and torch.isfinite(v).all()
        a, v, _ = pol(torch.from_numpy(x.reshape(5, 80)).float(), deterministic=True)
        a_ref, v_ref = _sb3_mlp_forward(sd, x.reshape(5, 80))
        assert np.allclose(a.detach().numpy(), a_ref, rtol=0, atol=1e-5) and np.allclose(v.detach().numpy(), v_ref, rtol=0, atol=1e-5)


def _sb3_mlp_policy_state(rng, obs_dim, action_dim, use_sde):
    """policy.pth of SB3's ActorCriticPolicy as A2C / PPO save it with the reference's defaults, filled with seeded
    values: FlattenExtractor (no parameters), net_arch pi=[64, 64] / vf=[64, 64] as Sequential(Linear, Tanh, Linear, Tanh),
    the action_net / value_net heads, log_std [action_dim] (diagonal Gaussian) or [64, action_dim] (gSDE, full_std)."""
    shapes = {"log_std": (64, action_dim) if use_sde else (action_dim,)}
    for tower in ("policy_net", "value_net"):
        shapes.update({f"mlp_extractor.{tower}.0.weight": (64, obs_dim), f"mlp_extractor.{tower}.0.bias": (64,),
                       f"mlp_extractor.{tower}.2.weight": (64, 64), f"mlp_extractor.{tower}.2.bias": (64,)})
    shapes.update({"action_net.weight": (action_dim, 64), "action_net.bias": (action_dim,),
                   "value_net.weight": (1, 64), "value_net.bias": (1,)})
    return {k: torch.from_numpy(rng.uniform(-0.3, 0.3, s).astype(np.float32)) for k, s in shapes.items()}


def _sb3_mlp_forward(sd, x):
    """Deterministic action (the Gaussian mean) and value of SB3's MlpPolicy for flattened observations, float64."""
    p = {k: v.double().numpy() for k, v in sd.items()}

    def tower(name):
        h = np.tanh(x @ p[f"mlp_extractor.{name}.0.weight"].T + p[f"mlp_extractor.{name}.0.bias"])
        return np.tanh(h @ p[f"mlp_extractor.{name}.2.weight"].T + p[f"mlp_extractor.{name}.2.bias"])
    return tower("policy_net") @ p["action_net.weight"].T + p["action_net.bias"], \
        (tower("value_net") @ p["value_net.weight"].T + p["value_net.bias"])[:, 0]


def _write_sb3_layout_zip(path, state_dict, use_sde, hyper):
    """A checkpoint in the member layout and `data` format of Stable-Baselines3's `model.save` (gymnasium Box spaces;
    the cloudpickled class and schedule entries stand in as opaque strings)."""
    import io
    import json
    import zipfile

    def box(shape, low, high):
        return {":type:": "<class 'gymnasium.spaces.box.Box'>", ":serialized:": "gAWV-opaque-", "dtype": "float32",
                "_shape": list(shape), "low_repr": low, "high_repr": high, "_np_random": None}
    data = {"policy_class": {":type:": "<class 'abc.ABCMeta'>", ":serialized:": "gAWV-opaque-",
                             "__module__": "stable_baselines3.common.policies"},
            "observation_space": box((10, 8), "-inf", "inf"), "action_space": box((1,), "-1.0", "1.0"),
            "lr_schedule": {":type:": "<class 'function'>", ":serialized:": "gAWV-opaque-"},
            "use_sde": use_sde, "sde_sample_freq": -1, "gamma": 0.99, "n_envs": 1, **hyper}
    buf = io.BytesIO()
    torch.save(state_dict, buf)
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED) as z:
        z.writestr("data", json.dumps(data, indent=4))
        z.writestr("policy.pth", buf.getvalue())
        z.writestr("_stable_baselines3_version", "2.3.2")


def test_evaluation_harness_cpu():
    from mpc_rl_for_avs_b200 import evaluation
    from mpc_rl_for_avs_b200.rl import A2CMPC, BatchedIntersectionEnv
    make_env = lambda: BatchedIntersectionEnv(16, 9, device="cpu", seed=11, duration_steps=40)   # noqa: E731
    stub = _StubMPC()
    algo = A2CMPC(make_env(), stub, n_steps=2)
    res = evaluation.compare({"pure_mpc": evaluation.pure_mpc_controller(stub),
                              "mpcrl": evaluation.mpcrl_controller(algo)}, make_env, n_episodes=40, max_steps=30)
    for r in res.values():
        assert r["episodes"] == 48 and 0 <= r["success_rate"] <= 1 and 0 <= r["collision_rate"] <= 1   # ceil(40 / 16) = 3 complete episodes per environment
        assert 1 <= r["avg_steps"] <= 30 and abs(r["avg_time"] - r["avg_steps"] * 0.1) < 1e-6 and r["avg_speed"] > 0
    # same seeds -> same numbers
    again = evaluation.evaluate(evaluation.pure_mpc_controller(stub), make_env(), 40, 30)
    assert again == res["pure_mpc"]


@pytest.mark.gpu
def test_a2c_mpc_in_the_loop_gpu():
    import mpc_rl_for_avs_b200 as pkg
    from mpc_rl_for_avs_b200.rl import A2CMPC, BatchedIntersectionEnv
    B = 256
    env = BatchedIntersectionEnv(B, 9, device="cuda", seed=5)
    mpc = pkg.BatchedPureMPC({"horizon": 16, "weight_speed": 1, "weight_control": 1, "weight_input_diff": 1},
                             vehicles_count=10, max_batch=B, collision_check=True)
    algo = A2CMPC(env, mpc, n_steps=8)
    for _ in range(2):
        log = algo.train_step()
    assert all(np.isfinite(v) for v in log.values())
    assert algo.stats["steps"] == 2 * 8 * B and algo.stats["mpc_s"] > 0
    # the latch of finished environments was cleared through reset_mask
    assert int(mpc.collision_memory[:B].max()) <= 10


@pytest.mark.gpu
def test_ppo_mpc_and_evaluation_gpu():
    import mpc_rl_for_avs_b200 as pkg
    from mpc_rl_for_avs_b200 import evaluation
    from mpc_rl_for_avs_b200.rl import PPOMPC, BatchedIntersectionEnv
    B = 256
    cfg = {"horizon": 16, "weight_speed": 1, "weight_control": 1, "weight_input_diff": 1}
    mpc = pkg.BatchedPureMPC(cfg, vehicles_count=10, max_batch=B, collision_check=True)
    algo = PPOMPC(BatchedIntersectionEnv(B, 9, device="cuda", seed=5), mpc, n_steps=8, n_epochs=2, batch_size=512)
    log = algo.train_step()
    assert all(np.isfinite(v) for v in log.values())
    make_env = lambda: BatchedIntersectionEnv(B, 9, device="cuda", seed=6, duration_steps=150)   # noqa: E731
    res = evaluation.compare({"pure_mpc": evaluation.pure_mpc_controller(mpc), "mpcrl": evaluation.mpcrl_controller(algo)},
                             make_env, n_episodes=B, max_steps=150)
    assert res["pure_mpc"]["episodes"] == B and res["mpcrl"]["episodes"] == B
    # the collision-aware MPC on the raw action path drives: it moves and most episodes end without a crash
    assert res["pure_mpc"]["avg_speed"] > 1.0 and res["pure_mpc"]["collision_rate"] < 0.6


@pytest.mark.gpu
def test_graph_captured_rollout_gpu():
    """The policy -> MPC -> env transition replayed from a CUDA graph fills the same buffers as the eager loop."""
    import mpc_rl_for_avs_b200 as pkg
    from mpc_rl_for_avs_b200.rl import A2CMPC, PPOMPC, BatchedIntersectionEnv
    B, T = 512, 12
    cfg = {"horizon": 16, "weight_speed": 1, "weight_control": 1, "weight_input_diff": 1}
    for Algo in (A2CMPC, PPOMPC):
        mpc = pkg.BatchedPureMPC(cfg, vehicles_count=10, max_batch=B, collision_check=True)
        algo = Algo(BatchedIntersectionEnv(B, 9, device="cuda", seed=9, duration_steps=20), mpc, n_steps=T, graph=True)
        ptrs, thetas = [], []
        for _ in range(3):
            log = algo.train_step()
            if algo.policy.use_sde:                      # gSDE (PPO default): the graph reads the noise buffer by address
                ptrs.append(algo.policy._theta.data_ptr())
                thetas.append(algo.policy._theta.clone())
        assert algo._cuda_graph is not None and all(np.isfinite(v) for v in log.values())
        if algo.policy.use_sde:
            assert len(set(ptrs)) == 1 and tuple(algo.policy._theta.shape) == (B, 64, 1)      # never re-bound by the update loop
            assert not torch.equal(thetas[0], thetas[1]) and not torch.equal(thetas[1], thetas[2])   # resampled per rollout
            with pytest.raises(RuntimeError):
                algo.policy.reset_noise(B // 2)         # would re-bind storage a captured graph still reads
        assert int(algo._row) == T and algo.num_timesteps == 3 * B * T
        obs_buf, buf = algo._obs_buf, algo._buf
        assert (obs_buf[:, :, 0] == 1).all() and torch.isfinite(obs_buf).all()         # every row written (presence flag of the ego)
        assert (obs_buf[1:] != obs_buf[:-1]).any(dim=-1).all()                          # the scene moves every step
        assert 0.0 < float(buf["done"].mean()) < 0.5                                    # 20-step episodes end inside the rollout
        assert torch.isfinite(buf["rew"]).all() and float(buf["act"].abs().max()) > 0
        # the MPC really ran inside the graph: fresh iteration counts and bounded actions
        assert int(mpc.iters[:B].max()) > 0 and float(mpc.actions[:B, 0].abs().max()) <= 5.0 + 1e-5
        assert int(mpc.collision_memory[:B].max()) <= 10


@pytest.mark.gpu
def test_fused_env_step_matches_the_tensor_program_gpu():
    """csrc/mpc_env.cu (one kernel per step) against the tensor program it restates: same seed, same actions ->
    same events and the same random respawns; states agree to float rounding."""
    from mpc_rl_for_avs_b200.rl import BatchedIntersectionEnv
    B = 1024
    a = BatchedIntersectionEnv(B, 9, device="cuda", seed=21, duration_steps=25, fused=True)
    b = BatchedIntersectionEnv(B, 9, device="cuda", seed=21, duration_steps=25, fused=False)
    assert a.fused and not b.fused and torch.equal(a.observe(), b.observe())
    gen = torch.Generator(device="cuda").manual_seed(3)
    n_done = n_crash = n_arrive = 0
    for step in range(60):
        act = torch.rand(B, 2, generator=gen, device="cuda") * 2.4 - 1.2
        act[:, 1] *= 0.2
        if step == 10:                                           # put a few egos just before the end of the path: arrivals
            for env in (a, b):
                env.ego[:32, 0] = env.ref_xy[-2, 0] + 0.5
                env.ego[:32, 1] = env.ref_xy[-1, 1]
                env.ego[:32, 2] = -math.pi
                env.ego[:32, 3] = 8.0
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        same = (da == db) & (ia["crashed"] == ib["crashed"]) & (ia["arrived"] == ib["arrived"])
        assert float(same.float().mean()) > 0.999, step        # an event can flip only on a rounding tie (2.5 m / arrival line)
        if not bool(same.all()):                                # re-synchronise the rare tie so the comparison can go on
            b.ego.copy_(a.ego); b.oth.copy_(a.oth); b.t.copy_(a.t); ob = oa
        assert torch.allclose(oa[same], ob[same], atol=2e-3, rtol=1e-4), step
        assert torch.allclose(ra[same], rb[same], atol=1e-4) and torch.equal(ia["truncated"][same], ib["truncated"][same])
        assert torch.allclose(ia["terminal_observation"][same], ib["terminal_observation"][same], atol=2e-3, rtol=1e-4)
        assert torch.equal(a._ctr, b._ctr) and torch.equal(a.t[same], b.t[same])
        n_done += int(da.sum()); n_crash += int(ia["crashed"].sum()); n_arrive += int(ia["arrived"].sum())
    assert n_done > B and n_crash > 0 and n_arrive > 0          # resets, crashes and arrivals were all exercised


@pytest.mark.gpu
def test_reference_signature_wrappers_gpu():
    """`A2C_MPC` / `PPO_MPC` with the reference's constructor keywords (agents/a2c_mpc.py:53-109, agents/ppo_mpc.py:94-200)
    and method names, n_envs > 1."""
    from mpc_rl_for_avs_b200.rl import A2C_MPC, PPO_MPC, BatchedIntersectionEnv
    B = 128
    pure_mpc_cfg = {"horizon": 16, "render": False, "weight_speed": 1, "weight_control": 1, "weight_input_diff": 1, "speed_override": 0}
    a2c = A2C_MPC(mpcrl_cfg={"action_space_dim": 1}, version="v0", pure_mpc_cfg=pure_mpc_cfg, policy="MlpPolicy",
                  env=BatchedIntersectionEnv(B, 9, device="cuda", seed=3), learning_rate=7e-4, n_steps=4, gae_lambda=1.0, verbose=0)
    a2c.learn(total_timesteps=2 * B * 4)
    assert a2c.num_timesteps == 2 * B * 4 and a2c.mpc_agent.n_obstacles == 9 and np.isfinite(a2c.last_log["loss"])
    ppo = PPO_MPC(mpcrl_cfg={"action_space_dim": 3}, version="v1", pure_mpc_cfg=pure_mpc_cfg, policy="MlpPolicy",
                  env=BatchedIntersectionEnv(B, 9, device="cuda", seed=4), use_collision_avoidance=False, n_steps=4, batch_size=64, n_epochs=2)
    ppo.train()
    assert ppo.num_timesteps == B * 4 and not ppo.mpc_agent.collision_check and np.isfinite(ppo.last_log["loss"])
    with pytest.raises(NotImplementedError):
        A2C_MPC({}, "v0", pure_mpc_cfg, "CnnPolicy", BatchedIntersectionEnv(B, 9, device="cuda", seed=3))
