"""The opt-in adaptive start portfolio (mpc_set_adaptive_starts / BatchedPureMPC.set_adaptive_starts).

A problem runs its base starts 0..S0-1; when they disagree (an objective not finite, or max - min > rel_gap *
max(|min|, 1)) it also runs starts S0..S-1 inside the same launch.  Its result must then be bit-identical to a fixed
S-start handle, and every other problem's to a fixed S0-start handle.  The CPU tests apply the rule to the host build's
per-start results on the golden sets; the GPU tests check the property on the device kernels."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import helpers

S0, S, GAP = 4, 8, 1e-3


# ----------------------------------------------------------------------------- the rule, in float32 like the kernel
def extend_rule(cost, n_base, rel_gap):
    """cost [>= n_base, B] float32 -> bool [B]."""
    c = np.asarray(cost[:n_base], dtype=np.float32)
    lo, hi = c.min(axis=0), c.max(axis=0)
    return ~np.all(np.isfinite(c), axis=0) | ((hi - lo) > np.float32(rel_gap) * np.maximum(np.abs(lo), np.float32(1)))


def select(cost, n):
    """k_select: lowest objective wins, ties to the lowest start, a NaN start 0 is replaced by any finite start."""
    best = np.zeros(cost.shape[1], int)
    Jb = cost[0].copy()
    for st in range(1, n):
        J = cost[st]
        take = (J < Jb) | (~(Jb == Jb) & (J == J))
        best[take], Jb[take] = st, J[take]
    return best, Jb


@pytest.fixture(scope="module")
def hs_starts():
    """tests/hostsim/hostsim_starts.cpp (the host harness plus hs_solve_starts), built into a temporary directory."""
    src = os.path.join(helpers.ROOT, "tests", "hostsim", "hostsim_starts.cpp")
    with tempfile.TemporaryDirectory() as tmp:
        so = os.path.join(tmp, "libhostsim_starts.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src])
        lib = C.CDLL(so)
    assert lib.hs_sizeof_config() == C.sizeof(helpers.HsConfig)
    return lib


def hostsim_starts(lib, d, cfg, n_starts):
    """hs_solve_starts: every start's cost, status, iterations and first control, [n_starts][B]."""
    P = C.POINTER
    B = d["ego_index"].shape[0]
    cost = np.zeros((n_starts, B), np.float32); st = np.zeros((n_starts, B), np.int32)
    it = np.zeros((n_starts, B), np.int32); u0 = np.zeros((n_starts, B, 2), np.float32)
    b = helpers._as_struct(d)
    f = lambda a, t: a.ctypes.data_as(P(t))  # noqa: E731
    lib.hs_solve_starts(C.byref(cfg), helpers.REF.ctypes.data_as(P(C.c_double)), C.byref(b), B, n_starts, f(cost, C.c_float),
                        f(st, C.c_int), f(it, C.c_int), f(u0, C.c_float))
    return cost, st, it, u0


SETS = [("golden_track", 0, 0.0), ("golden_coll", 8, 10.0), ("golden_holdout", 8, 10.0), ("golden_holdout_1k", 8, 10.0)]
# host build of the device code, rel_gap 1e-3, measured: extended fraction 19.5 % / 19.5 % / 25.0 % / 23.6 %, i.e.
# 4.78 / 4.78 / 5.00 / 4.95 starts per problem; J_gpu <= J_oracle (all) fixed 4 / adaptive / fixed 8:
# 89.5 / 89.8 / 90.6 %, 91.0 / 91.8 / 92.2 %, 88.3 / 88.7 / 88.7 %, 87.6 / 88.6 / 89.0 %; in-path 97.6 / 98.1 / 98.6 %,
# 99.0 / 99.5 / 100 %, 93.7 / 94.1 / 94.1 %, 95.6 / 96.6 / 97.1 %.  The first control within 1e-3 of the best known
# optimum moves by at most 1 % either way (also between fixed 4 and fixed 8: a lower objective is not always the same
# optimum as the yardstick's).
MAX_MEAN_STARTS = 5.1
BARS = {"golden_track": dict(below=0.89, in_path=0.97), "golden_coll": dict(below=0.91, in_path=0.99),
        "golden_holdout": dict(below=0.88, in_path=0.93), "golden_holdout_1k": dict(below=0.88, in_path=0.96)}


def _golden(name):
    g = helpers.load_golden(name)
    d = {k[len("batch_"):]: v for k, v in g.items() if k.startswith("batch_")}
    return g, d


def test_hostsim_starts_reproduce_the_portfolio_winners(hs_starts):
    hostsim = hs_starts
    g, d = _golden("golden_coll")
    cfg = helpers.hs_config(M=8, w_distance=10.0)
    cost, st, it, u0 = hostsim_starts(hostsim, d, cfg, S)
    ar = np.arange(cost.shape[1])
    for n in (S0, S):
        r = helpers.hostsim_solve_init(hostsim, d, cfg, n_starts=n)
        best, Jb = select(cost, n)
        assert np.array_equal(Jb.view(np.int32), r["cost"].view(np.int32))
        assert np.array_equal(u0[best, ar], r["actions"])
        assert np.array_equal(st[best, ar], r["status"])
        assert np.array_equal(it[:n].sum(axis=0), r["iters"])


@pytest.mark.parametrize("name,M,wd", SETS)
def test_rule_on_golden_sets(hs_starts, name, M, wd):
    """The adaptive result is the fixed-8 result where the rule extends and the fixed-4 result elsewhere."""
    hostsim = hs_starts
    g, d = _golden(name)
    cfg = helpers.hs_config(M=M, w_distance=wd)
    probs, _ = helpers.problems_from_obs(g["obs"], g["ref_speed"], g["has_ref_speed"], w_distance=float(g["w_distance"]),
                                         collision_check=bool(g["collision_check"]))
    cost, _, _, _ = hostsim_starts(hostsim, d, cfg, S)
    r4 = helpers.hostsim_solve_init(hostsim, d, cfg, n_starts=S0)
    r8 = helpers.hostsim_solve_init(hostsim, d, cfg, n_starts=S)
    ext = extend_rule(cost, S0, GAP)
    ra = {k: np.where(ext.reshape((-1,) + (1,) * (v.ndim - 1)), r8[k], v) for k, v in r4.items()}
    assert S0 + (S - S0) * ext.mean() <= MAX_MEAN_STARTS
    s4, sa, s8 = (helpers.solve_parity_stats(r, g, probs) for r in (r4, ra, r8))
    for tag in ("all", "in_path"):
        assert sa[tag]["below"] >= s4[tag]["below"], (tag, sa[tag], s4[tag])
        assert sa[tag]["below"] >= s8[tag]["below"] - 0.01, (tag, sa[tag], s8[tag])
        assert abs(sa[tag]["same"] - s4[tag]["same"]) <= 0.01 and abs(sa[tag]["same"] - s8[tag]["same"]) <= 0.01, tag
    assert sa["all"]["below"] >= BARS[name]["below"] and sa["in_path"]["below"] >= BARS[name]["in_path"], sa


def test_set_adaptive_starts_rejects_a_null_handle():
    from mpc_rl_for_avs_b200 import _capi
    lib = _capi.load()
    assert lib.mpc_set_adaptive_starts(None, 8, 1e-3, None, None) == _capi.ERR_BAD_ARG


# ----------------------------------------------------------------------------- on the B200
CFG = {"horizon": 20, "weight_speed": 1.0, "weight_control": 1.0, "weight_input_diff": 1.0}
M = 8


def _pkg():
    import mpc_rl_for_avs_b200 as pkg
    return pkg


def _config3(B, seed=1234):
    """bench.py's config-3 inputs: 8 obstacles, RL reference speed on half of the batch (NaN = none)."""
    import torch
    obs, rs, has = _pkg().make_scenarios(B, M, seed=seed)
    rsn = torch.where(has.reshape(-1, 1), rs, torch.full_like(rs, float("nan"))).reshape(-1).contiguous()
    return obs.cuda(), rsn.cuda()


def _agent(max_batch, n_starts, tpb=0, adaptive=None):
    a = _pkg().BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=max_batch, collision_check=True, weight_distance=10.0,
                              n_starts=n_starts, threads_per_block=tpb)
    if adaptive is not None:
        a.set_adaptive_starts(S, adaptive)
    return a


def _solve(agent, obs, rs, B):
    import torch
    agent.reset()
    a, U = agent.predict_batch(obs[:B].contiguous(), ref_speed=rs[:B].contiguous(), return_controls=True)
    torch.cuda.synchronize()
    r = dict(actions=a.clone(), status=agent.status[:B].clone(), cost=agent.cost[:B].clone(), U=U.clone(),
             iters=agent.iters[:B].clone())
    if agent.max_starts:
        r["start_cost"] = agent.start_cost[:, :B].clone()
        r["extended"] = agent.extended[:B].clone().bool()
    return r


def _bits(t):
    import torch
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_by_extension(ra, r4, r8, ext):
    for k in ("actions", "status", "cost", "U", "iters"):
        a, f4, f8 = _bits(ra[k]), _bits(r4[k]), _bits(r8[k])
        m = ext.reshape((-1,) + (1,) * (a.dim() - 1)).expand_as(a)
        assert bool((a[m] == f8[m]).all()), ("extended", k)
        assert bool((a[~m] == f4[~m]).all()), ("base", k)


def _assert_same(x, y):
    for k in x:
        assert bool((_bits(x[k]) == _bits(y[k])).all()), k


@pytest.mark.gpu
def test_bit_exact_against_fixed_portfolios():
    import torch
    B = 8192
    obs, rs = _config3(B)
    r4, r8 = _solve(_agent(B, S0), obs, rs, B), _solve(_agent(B, S), obs, rs, B)
    ra = _solve(_agent(B, S0, adaptive=GAP), obs, rs, B)
    ext = ra["extended"]
    rule = extend_rule(ra["start_cost"].cpu().numpy(), S0, GAP)
    assert np.array_equal(ext.cpu().numpy(), rule)
    assert 0.05 < float(ext.float().mean()) < 0.6
    _assert_by_extension(ra, r4, r8, ext)
    sc = ra["start_cost"]
    assert bool(torch.isnan(sc[S0:, ~ext]).all())
    assert not bool(torch.isnan(sc[:S0]).all(dim=0).any())
    # the returned objective is the lowest of the starts that ran
    low = torch.where(torch.isnan(sc), torch.full_like(sc, float("inf")), sc).amin(dim=0)
    ok = torch.isfinite(ra["cost"])
    assert bool((low[ok] == ra["cost"][ok]).all())


@pytest.mark.gpu
def test_limits_of_rel_gap():
    import torch
    B = 8192
    obs, rs = _config3(B, seed=2234)
    r4, r8 = _solve(_agent(B, S0), obs, rs, B), _solve(_agent(B, S), obs, rs, B)
    ag = _agent(B, S0, adaptive=math.inf)
    ra = _solve(ag, obs, rs, B)
    nonfinite = torch.from_numpy(~np.all(np.isfinite(ra["start_cost"][:S0].cpu().numpy()), axis=0)).to(ra["extended"].device)
    assert torch.equal(ra["extended"], nonfinite)            # +inf: only a non-finite base objective extends
    _assert_by_extension(ra, r4, r8, ra["extended"])
    ag.set_adaptive_starts(S, -1.0)
    ra = _solve(ag, obs, rs, B)
    assert bool(ra["extended"].all())
    _assert_same({k: ra[k] for k in r8}, r8)


@pytest.mark.gpu
@pytest.mark.parametrize("tpb", [128, 192, 256, 64])
def test_repeatable_under_every_kernel(tpb):
    """Forced TMEM blocks (128 without compaction, 192/256 with compaction and speculation) and the shared-memory gains
    kernel k_solve<64>: two adaptive launches are bit-identical, and match fixed runs of the same kernel."""
    Bmax = 65536
    obs, rs = _config3(Bmax, seed=3234)
    f4, f8, ad = _agent(Bmax, S0, tpb), _agent(Bmax, S, tpb), _agent(Bmax, S0, tpb, adaptive=GAP)
    sc = ad.solve_config(Bmax)
    assert sc["threads_per_block"] == tpb and sc["gains_in_tmem"] == (tpb >= 128)
    for B in (1, 37, 4096, 65536):
        ra, rb = _solve(ad, obs, rs, B), _solve(ad, obs, rs, B)
        _assert_same(ra, rb)
        _assert_by_extension(ra, _solve(f4, obs, rs, B), _solve(f8, obs, rs, B), ra["extended"])


@pytest.mark.gpu
def test_switching_off_restores_the_fixed_portfolio():
    B = 4096
    obs, rs = _config3(B, seed=4234)
    ad = _agent(B, S0, adaptive=GAP)
    _solve(ad, obs, rs, B)
    ad.set_adaptive_starts(None)
    assert ad.start_cost is None and ad.extended is None
    _assert_same(_solve(ad, obs, rs, B), _solve(_agent(B, S0), obs, rs, B))


@pytest.mark.gpu
def test_with_a_warm_start():
    B = 4096
    obs, rs = _config3(B, seed=5234)
    f4, f8, ad = _agent(B, S0), _agent(B, S), _agent(B, S0, adaptive=GAP)
    U0 = f4.shift_controls(_solve(f4, obs, rs, B)["U"])
    for a in (f4, f8, ad):
        a.set_warm_start(U0)
    ra = _solve(ad, obs, rs, B)
    _assert_by_extension(ra, _solve(f4, obs, rs, B), _solve(f8, obs, rs, B), ra["extended"])


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager():
    import torch
    B = 4096
    obs, rs = _config3(B, seed=6234)
    ad = _agent(B, S0, adaptive=GAP)
    eager = _solve(ad, obs, rs, B)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ad.reset()
        ad.predict_batch(obs, ref_speed=rs)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ad.predict_batch(obs, ref_speed=rs)
    for _ in range(2):
        ad.reset()
        ad.start_cost.zero_()
        ad.extended.fill_(7)
        g.replay()
        torch.cuda.synchronize()
        for k, v in (("actions", ad.actions[:B]), ("status", ad.status[:B]), ("cost", ad.cost[:B]), ("iters", ad.iters[:B]),
                     ("start_cost", ad.start_cost[:, :B]), ("extended", ad.extended[:B].bool())):
            assert bool((_bits(v) == _bits(eager[k])).all()), k


@pytest.mark.gpu
def test_bad_arguments_raise():
    ad = _agent(64, S0)
    for bad in (0 + S0, S0 - 1, 9):
        with pytest.raises(ValueError):
            ad.set_adaptive_starts(bad)
    with pytest.raises(ValueError):
        ad.set_adaptive_starts(S, float("nan"))
    with pytest.raises(ValueError):
        _agent(64, 1).set_adaptive_starts(S)
    from mpc_rl_for_avs_b200 import _capi
    lib = _capi.load()
    for ms, gap in ((S0, 1e-3), (9, 1e-3), (S, float("nan"))):
        assert lib.mpc_set_adaptive_starts(ad._h, ms, gap, None, None) == _capi.ERR_BAD_ARG
    one = _agent(64, 1)
    assert lib.mpc_set_adaptive_starts(one._h, S, 1e-3, None, None) == _capi.ERR_BAD_ARG
    # max_batch * max_starts past the limit of mpc_create (2^31 / 64 work items) while max_batch * n_starts is within it
    big = _pkg().BatchedPureMPC(CFG, vehicles_count=2, max_batch=1 << 22, collision_check=False, n_starts=S0)
    with pytest.raises(ValueError):
        big.set_adaptive_starts(S)
    assert lib.mpc_set_adaptive_starts(big._h, S, 1e-3, None, None) == _capi.ERR_BAD_ARG
    assert lib.mpc_set_adaptive_starts(big._h, S0 + 1, 1e-3, None, None) == 0
