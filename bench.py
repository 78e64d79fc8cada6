"""bench.py -- MPC solves/sec (H=20, 8 obstacles) on B200.  See DESIGN.md "Measurement".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--n-starts S] [--config 1|2|3]
                  [--dump-outputs DIR]

--config 3 (default) is the headline workload; the same JSON line carries the other BASELINE configurations as extra
keys (`single_start`, `config1_latency`, `config2`, and `config5` under --gpus N); --config 1 / 2 print only that one.
--steps K sets the number of timed steps of every measurement except config 1 (--config 1 and the `config1_latency`
key), whose timed region is the workload itself: the 100-call closed loop of the reference's run script.

--dump-outputs DIR saves what the last timed step of the config-3 path computed (actions, cost, status, is_collide); the
inputs depend only on the arguments, so two builds run with the same arguments can be compared output for output.
Under --gpus N rank 0 writes its own shard: cost, status and is_collide exist only on the rank that solved those
problems, and rank 0's part of the gathered actions is its local actions.  Configs 1 and 2 and --impl reference are
not dumped (--dump-outputs is refused there).

One "step" = one full predict (parse -> collision check -> regeneration -> solve to convergence ->
first control) over one batch of synthetic intersection scenarios (BASELINE config 3: 65536
problems, H=20, 8 obstacles, distance cost 10, collision check + regeneration).  Every step uses a
fresh, different batch (seeded), with the latch cleared.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("OMP_NUM_THREADS", "1")

H, M, W_DIST = 20, 8, 10.0
CFG = {"horizon": H, "weight_speed": 1.0, "weight_control": 1.0, "weight_input_diff": 1.0}
WORKLOAD = "config3: 65536 synthetic intersection problems/GPU, H=20, 8 obstacles, distance cost 10, collision check + ref-speed regeneration"


def workload(batch: int) -> str:
    return WORKLOAD if batch == 65536 else WORKLOAD.replace("65536", str(batch)) + " (non-default --batch)"


def flops_per_solve(mean_iters: float, m: int = M, h: int = H, latched_frac: float = 0.0) -> float:
    """SURVEY 8-d yardstick: F_solve = I*H*(960+47M) + 18.7k*M per un-latched collision check."""
    return mean_iters * h * (960 + 47 * m) + (1.0 - latched_frac) * 18.7e3 * m


class ClockSampler:
    def __init__(self, gpu_index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._idx = gpu_index
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._idx)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
            while not self._stop.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.01)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def start(self):
        self._t.start()

    def stop(self):
        self._stop.set()
        self._t.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def run_reference(args) -> None:
    """The reference's CPU path for the same workload: the FP64 oracle (casadi/shapely are not
    installable, so `oracle/_ref` does not exist -- kind "port"), one problem per call as the reference
    is used (agents/a2c_mpc.py:145-150), on every host core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import multiprocessing as mp
    import numpy as np
    import mpc_rl_for_avs_b200 as pkg
    cores = os.cpu_count() or 1
    per_step = args.ref_problems if args.ref_problems > 0 else 24 * cores
    obs, rs, has = pkg.make_scenarios(per_step * (args.steps + args.warmup), M, seed=1234)
    obs, rs, has = obs.numpy(), rs.numpy(), has.numpy()
    items = [(obs[i], (rs[i] if has[i] else None)) for i in range(obs.shape[0])]
    with mp.Pool(cores) as pool:
        pool.map(_ref_one, items[: per_step * args.warmup], chunksize=1)
        t0 = time.perf_counter()
        pool.map(_ref_one, items[per_step * args.warmup:], chunksize=1)
        dt = time.perf_counter() - t0
    n = per_step * args.steps
    v = n / dt
    line = {"impl": "reference", "metric": "mpc_solves_per_sec", "value": v, "unit": "solves/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sampled": True, "problems": per_step,
                       "sample": f"{per_step} problems/step of the same seeded workload (throughput is per problem)"},
            "cpu_baseline": {"value": v, "unit": "solves/s", "cores": cores, "kind": "port",
                             "sample": f"{n} problems of the same seeded workload, one per task over {cores} processes"},
            "e2e": {"value": v, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def _ref_one(item):
    import numpy as np
    import mpc_oracle as orc
    obs, r = item
    ag = orc.OraclePureMPCAgent(horizon=H, vehicles_count=M + 1, weight_distance=W_DIST, collision_check=True)
    u0 = ag.predict(obs, ref_speed=None if r is None else np.asarray(r).reshape(1, 1))
    # the cost that is compared with the device's is the cost of a FEASIBLE point: SLSQP honours the node bounds only
    # to its tolerance (the timed region is the predict call above; this is bookkeeping of the parity sample)
    feas = orc.objective(orc.repair_feasible(ag.last_solution.U, ag.last_problem), ag.last_problem)
    return u0[0], u0[1], feas


def _cost64(item):
    """FP64 objective of given controls for one scene (oracle as checker)."""
    import numpy as np
    import mpc_oracle as orc
    obs, r, U = item
    ag = orc.OraclePureMPCAgent(horizon=H, vehicles_count=M + 1, weight_distance=W_DIST, collision_check=True)
    parsed = orc.parse_obs(obs, M + 1)
    ag.check_collision(parsed)
    prob = ag.build_problem(parsed, None, None if r is None else np.asarray(r).reshape(1, 1))
    return orc.objective(np.asarray(U, dtype=np.float64), prob)


def _confirm(item):
    """The tests' optimality check (tests/helpers.py: oracle_warm_confirms) for one scene: SLSQP started at the device's
    controls, pulled back into the feasible set, must neither move the first control by 1e-3 nor gain 1e-6 relative."""
    import numpy as np
    import mpc_oracle as orc
    obs, r, U = item
    ag = orc.OraclePureMPCAgent(horizon=H, vehicles_count=M + 1, weight_distance=W_DIST, collision_check=True)
    parsed = orc.parse_obs(obs, M + 1)
    ag.check_collision(parsed)
    prob = ag.build_problem(parsed, None, None if r is None else np.asarray(r).reshape(1, 1))
    U = np.asarray(U, dtype=np.float64)
    c0 = orc.objective(U, prob)
    Us = orc.repair_feasible(orc.solve_nlp(prob, U0=U).U, prob)
    gain = (c0 - orc.objective(Us, prob)) / (1.0 + abs(c0))
    gain_ok = gain < 1e-6
    stays = np.max(np.abs(Us[0] - U[0])) < 1e-3 or gain < 4 * 1.1920929e-7     # a valley below FP32 rounding of J is not a disagreement
    return bool(stays and gain_ok)


class _StubEnv:
    """Closed-loop stand-in for main/run_pure_mpc.py's env (highway-env is not installable): bicycle ego at the policy
    rate with the script's action scaling, straight-driving others."""
    config = {"simulation_frequency": 30, "policy_frequency": 10, "observation": {"vehicles_count": M + 1}}

    def __init__(self, seed=0):
        import mpc_rl_for_avs_b200 as pkg
        self.unwrapped = self
        self.obs0 = pkg.make_scenarios(1, M, seed=4000 + seed)[0][0].numpy().copy()

    def reset(self):
        import numpy as np
        self.o = self.obs0.astype(np.float64)
        self.o[0, 1:3] = (2.0, 49.0)
        self.o[0, 5] = -np.pi / 2
        self.v = 8.0
        return self._obs(), {}

    def _obs(self):
        import numpy as np
        th = self.o[0, 5]
        self.o[0, 3:5] = (self.v * np.cos(th), self.v * np.sin(th))
        self.o[0, 6:8] = (np.sin(th), np.cos(th))
        return self.o.astype(np.float32)

    def step(self, action):
        import numpy as np
        a, d = 5.0 * float(np.clip(action[0], -1, 1)), (np.pi / 4) * float(np.clip(action[1], -1, 1))
        beta = np.arctan(0.5 * np.tan(d))
        th = self.o[0, 5]
        self.o[0, 1] += 0.1 * self.v * np.cos(th + beta)
        self.o[0, 2] += 0.1 * self.v * np.sin(th + beta)
        self.o[0, 5] = th + 0.1 * self.v / 2.5 * np.sin(beta)
        self.v = max(self.v + 0.1 * a, 0.0)
        self.o[1:, 1:3] += 0.1 * self.o[1:, 3:5]
        return self._obs(), 0.0, False, False, {}


def config1_latency(pkg, device, n_starts=0, steps=100):
    """BASELINE config 1: one scenario through the PureMPC_Agent drop-in (B = 1), the closed 100-step loop of
    main/run_pure_mpc.py:25-30, wall-clock per predict() call including its host<->device copies."""
    import numpy as np
    cfg = {"horizon": H, "render": False, "weight_speed": 1, "weight_control": 1, "weight_input_diff": 1, "speed_override": 0}
    env = _StubEnv()
    agent = pkg.PureMPC_Agent(env, cfg, device=device, n_starts=n_starts)
    lat = []
    for rep in range(2):                 # first pass = warm-up
        obs, _ = env.reset()
        agent._solver.reset()
        agent.collision_memory, agent.memorized_conflict_points, agent.memorized_conflict_indices = 0, None, None
        lat = []
        import io, contextlib
        for _ in range(steps):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                act = agent.predict(obs, False)
            lat.append(time.perf_counter() - t0)
            obs, *_ = env.step([act.acceleration / 5, act.steer / (np.pi / 3)])
    lat = np.sort(np.array(lat)) * 1e3
    return {"workload": "config1: PureMPC_Agent.predict, B=1, 100-step closed loop (stub env), host numpy in/out",
            "p50_ms": float(lat[len(lat) // 2]), "p99_ms": float(lat[int(0.99 * (len(lat) - 1))]), "mean_ms": float(lat.mean()),
            "solves_per_sec": float(1e3 / lat.mean()), "n_starts": agent._solver.n_starts}


def timed_steps(torch, fn, steps, warmup=3):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


DUMP_LIMIT_BYTES = 64_000_000
NPY_HEADER_BYTES = 128          # the .npy header numpy writes for a short dtype / shape description


def dump_outputs(out_dir: str, tensors) -> None:
    """Saves per-problem outputs as float32 (status codes and flags are small integers, exact in float32).  When the
    files, headers included, would exceed DUMP_LIMIT_BYTES, a fixed seeded sample of problems is kept and its indices
    go to sample_index.npy (float64)."""
    import numpy as np
    arrays = {k: v.cpu().numpy().astype(np.float32) for k, v in tensors.items()}
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes + len(arrays) * NPY_HEADER_BYTES > DUMP_LIMIT_BYTES:
        row_bytes += 8                                                   # + sample_index
        n_keep = (DUMP_LIMIT_BYTES - (len(arrays) + 1) * NPY_HEADER_BYTES) // row_bytes
        idx = np.sort(np.random.default_rng(0).choice(n, n_keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["sample_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=65536, help="problems per GPU per step")
    ap.add_argument("--ref-problems", type=int, default=0, help="reference arm: problems per step")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--n-starts", type=int, default=0, help="start portfolio size (0 = library default, 4; 1 = the reference's cold start only)")
    ap.add_argument("--config", type=int, default=3, choices=(1, 2, 3), help="BASELINE configuration to print (3 = headline)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra keys (single_start, config1_latency, config2, config5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (actions, cost, status, is_collide; rank 0's shard) "
                         "as DIR/<name>.npy, for comparing the outputs of two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config != 3):
        ap.error("--dump-outputs applies to the config-3 path of --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import mpc_rl_for_avs_b200 as pkg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the MPC path has no CPU implementation")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    total = B * world
    tune = {k: int(os.environ[e]) for k, e in (("max_iter", "MPC_MAX_ITER"), ("threads_per_block", "MPC_TPB"),
                                                ("blocks_per_sm", "MPC_BPS")) if e in os.environ}      # experiments only
    if args.config == 1:
        if rank == 0:
            print(json.dumps({"metric": "mpc_predict_latency_ms", "unit": "ms", "higher_is_better": False, "n_gpus": 1,
                              **config1_latency(pkg, local, args.n_starts)}), flush=True)
        return
    if args.config == 2:
        if rank == 0:
            print(json.dumps({"metric": "mpc_solves_per_sec", "unit": "solves/s", "higher_is_better": True, "n_gpus": 1,
                              **config2(pkg, torch, local, args.n_starts, args.steps)}), flush=True)
        return
    agent = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=B, device=local, collision_check=True,
                               weight_distance=W_DIST, n_starts=args.n_starts, **tune)

    nsteps = args.warmup + args.steps
    # distinct batches per step; inputs live in HBM before the timed region (value) and in pinned host
    # memory (e2e).  Distinct data per step: nothing is cached between steps.
    n_unique = min(nsteps, 8)       # 8 x 19.4 MB of inputs > 126 MB L2
    batches = []
    for s in range(n_unique):
        obs, rs, has = pkg.make_scenarios(B, M, seed=1234 + rank + 1000 * s)
        rsn = torch.where(has.reshape(-1, 1), rs, torch.full_like(rs, float("nan"))).reshape(-1).contiguous()
        batches.append((obs.contiguous(), rsn))
    dev_batches = [(o.to(dev), r.to(dev)) for o, r in batches]
    host_batches = [(o.pin_memory(), r.pin_memory()) for o, r in batches]
    # two gathered-action buffers used alternately: k_solve writes this rank's actions straight into its slice, and the
    # in-place NCCL all-gather of step i runs on a side stream while k_prepare / k_solve of step i + 1 execute
    pipe = pkg.sharding.PipelinedActionGather(total, dev) if world > 1 else None
    gatherer = pipe.slots[0] if pipe is not None else None

    def step(i):
        o, r = dev_batches[i % n_unique]
        agent.reset()
        if pipe is not None:
            agent.bind_actions(pipe.acquire(i).local)
        a = agent.predict_batch(o, ref_speed=r)
        if pipe is not None:
            pipe.issue(i)                        # every rank ends up with all actions (pipe.result(i))
        return a

    def barrier():
        if pipe is not None:
            pipe.drain()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    iters_acc, conv_acc = [], []
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = agent.launch_count()
    agent.timing_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    if pipe is not None:
        pipe.drain()                             # the last all-gather belongs to the timed region
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    kt = agent.timing_end()
    launches = agent.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # taken before the e2e pass below reuses the agent's output buffers
        dump_outputs(args.dump_outputs, {"actions": agent.actions[:B], "cost": agent.cost[:B], "status": agent.status[:B],
                                         "is_collide": agent.is_collide[:B]})
    it = agent.iters[:B].float()
    st = agent.status[:B]
    mean_iters = float(it.mean())
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = total * args.steps / (ms * 1e-3)

    # ---- e2e: HOST buffers through the C-ABI host entry point (mpc_predict_host): pinned numpy in,
    # numpy out, H2D of obs/ref_speed/reset mask and D2H of actions/status/is_collide inside the call
    host_np = [(o.numpy(), r.numpy()) for o, r in host_batches]          # views of the pinned buffers
    reset_all = torch.ones(B, dtype=torch.uint8).pin_memory().numpy()
    h2d = d2h = 0

    def e2e_step(i):
        o, r = host_np[i % n_unique]
        acts, stat, iscol, up, down = agent.predict_host(o, r, reset_mask=reset_all)
        if gatherer is not None:
            gatherer.local.copy_(torch.from_numpy(acts), non_blocking=True)
            gatherer.gather()
        return up, down

    for i in range(3):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        h2d, d2h = e2e_step(i)
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = total * args.steps / float(t.item())

    # ---- BASELINE config 5: 2^20 problems of the same type sharded over the ranks, all-gather of the actions ----------
    config5 = None
    if world > 1 and not args.no_extras:
        B5 = (1 << 20) // world
        a5 = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=B5, device=local, collision_check=True,
                                weight_distance=W_DIST, n_starts=args.n_starts, **tune)
        g5 = pkg.sharding.PipelinedActionGather(B5 * world, dev)
        o5, rs5, has5 = pkg.make_scenarios(B5, M, seed=555 + rank)
        r5 = torch.where(has5.reshape(-1, 1), rs5, torch.full_like(rs5, float("nan"))).reshape(-1).contiguous().to(dev)
        o5 = o5.contiguous().to(dev)

        def s5(i):
            a5.reset()
            a5.bind_actions(g5.acquire(i).local)
            a5.predict_batch(o5, ref_speed=r5)
            g5.issue(i)
        s5(0)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for i in range(3):
            s5(i)
        g5.drain()
        c1.record()
        barrier()
        t5 = torch.tensor([c0.elapsed_time(c1) / 3], device=dev)
        dist.all_reduce(t5, op=dist.ReduceOp.MAX)
        config5 = {"workload": "config5: 2^20 collision-aware problems sharded over the ranks, all_gather(actions)",
                   "problems": B5 * world, "ms_per_sweep": float(t5.item()), "value": B5 * world / (float(t5.item()) * 1e-3), "unit": "solves/s"}
        a5.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (k_solve), FP32 non-tensor ------------------------------------
    sc = agent.solve_config(B)
    kernel_name = ("k_solve_tmem<%d>" if sc["gains_in_tmem"] else "k_solve<%d>") % sc["threads_per_block"]
    peak_tf = agent.fp32_peak_tflops(5)
    solve_ms = kt["solve_ms"]
    # mean_iters = iterations per problem summed over the starts of the portfolio: the algorithmic work of the launch
    alg_flops = flops_per_solve(mean_iters) * B - 18.7e3 * M * B      # collision-check flops belong to k_prepare
    achieved = alg_flops / (solve_ms * 1e-3) / 1e12 if solve_ms > 0 else 0.0
    hbm_bytes = (32 * M + 76) * B
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    traffic = None
    try:      # dram bytes read+written by k_solve per launch, from the committed `ncu --set full` capture of this command
        if B == 65536:       # the capture is of the default workload only
            for nm in ("r02_k_solve_ncu_full.json", "r01_k_solve_ncu_full.json"):
                pth = os.path.join(ROOT, "profiles", nm)
                if os.path.exists(pth):
                    traffic = json.load(open(pth))["dram_traffic_bytes_per_launch"]
                    break
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    roofline = {"bound": "fp32", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf if peak_tf else None,
                "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read+write; algorithmic %d)" % hbm_bytes, "kernel": kernel_name, "kernel_ms": solve_ms, "prepare_kernel_ms": kt["prepare_ms"],
                "kernel_share_of_step": (solve_ms * kt["n_solve"]) / ms if ms else None,
                "peak_source": "FP32 FMA micro-kernel measured in this run (mpc_fp32_peak); MEASURED_PEAKS.json holds only HBM/bf16",
                "alg_flops_per_launch": alg_flops, "mean_iters": mean_iters,
                "hbm": {"achieved_gbs": hbm_bytes / (solve_ms * 1e-3) / 1e9 if solve_ms else None, "peak_gbs": hbm_peak,
                        "frac": (hbm_bytes / (solve_ms * 1e-3) / 1e9) / hbm_peak if solve_ms else None,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}

    # ---- cpu_baseline: the oracle port on the host cores, bounded sample of the same workload -----------
    cpu = None
    if not args.no_cpu_baseline:
        cpu = cpu_baseline(args.cpu_seconds, agent if world == 1 else None)
    extras = {}
    if not args.no_extras:
        # the other BASELINE configurations, measured in the same run (device-resident inputs, CUDA events)
        if agent.n_starts != 1:
            a1 = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=B, device=local, collision_check=True,
                                    weight_distance=W_DIST, n_starts=1, **tune)

            def s1(i):
                o, r = dev_batches[i % n_unique]
                a1.reset()
                a1.predict_batch(o, ref_speed=r)
            ms1 = timed_steps(torch, s1, args.steps)
            st1 = a1.status[:B]
            extras["single_start"] = {"n_starts": 1, "value": B / (ms1 * 1e-3), "unit": "solves/s", "ms_per_step": ms1,
                                      "mean_iters": float(a1.iters[:B].float().mean()),
                                      "converged_frac": float((st1 == 0).float().mean()),
                                      "settled_frac": float(((st1 & ~32) == 0).float().mean()),
                                      "note": "only the reference's own cold start (zero controls, agents/pure_mpc.py:244)"}
            a1.close()
        if world == 1:
            extras["config1_latency"] = config1_latency(pkg, local, args.n_starts)
            extras["config2"] = config2(pkg, torch, local, args.n_starts, args.steps)

    line = {"metric": "mpc_solves_per_sec", "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload(B), "batch_per_gpu": B, "horizon": H, "obstacles": M,
                       "l2": "inputs rotate over 8 distinct batches (8 x 19.4 MB > the 126 MB L2); "
                             "the per-step working set is on-chip, HBM traffic is the compulsory ~0.3 KB/problem",
                       "parallelism": f"env-sharded x{world}" + (", all_gather(actions)" if world > 1 else "")},
            "solver": {"n_starts": agent.n_starts, "mean_iters": mean_iters, "p50_iters": float(it.median()), "p99_iters": float(torch.quantile(it, 0.99)),
                       "converged_frac": float((st == 0).float().mean()), "settled_frac": float(((st & ~32) == 0).float().mean()),
                       "kink_frac": float((st == 32).float().mean()), "max_iter_frac": float(((st & 1) != 0).float().mean()),
                       "note": "iterations are summed over the starts of the portfolio; converged = un-damped Newton test (status 0), "
                               "settled = converged or stationary on a kink of the clamped dynamics (status 32)"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "roofline": roofline, "cpu_baseline": cpu, **extras}
    if world > 1:
        line["config5"] = config5
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def config2(pkg, torch, device, n_starts, steps):
    """BASELINE config 2: 4096 problems, H=20, no collision logic, tracking objective (agents/pure_mpc.py:204-212 with
    the collision check off; the literal objective of pure_mpc_no_collision.py has u = 0 as its optimum, quirk Q3)."""
    B2 = 4096
    ag = pkg.BatchedPureMPC(CFG, vehicles_count=1, max_batch=B2, device=device, collision_check=False, n_starts=n_starts)
    obs, rs, has = pkg.make_scenarios(B2, 0, seed=51)
    rsn = torch.where(has.reshape(-1, 1), rs, torch.full_like(rs, float("nan"))).reshape(-1).contiguous().cuda(device)
    od = obs.contiguous().cuda(device)
    ms = timed_steps(torch, lambda i: ag.predict_batch(od, ref_speed=rsn), steps)
    st = ag.status[:B2]
    out = {"workload": "config2: 4096 synthetic problems, H=20, no collision logic, tracking objective", "value": B2 / (ms * 1e-3),
           "unit": "solves/s", "ms_per_step": ms, "n_starts": ag.n_starts, "mean_iters": float(ag.iters[:B2].float().mean()),
           "converged_frac": float((st == 0).float().mean()), "settled_frac": float(((st & ~32) == 0).float().mean())}
    ag.close()
    return out


def cpu_baseline(seconds: float, agent=None):
    """Oracle port on all host cores, one problem per task, first problems of the seeded workload.
    With `agent`, the same problems also go through the CUDA path (untimed) and the line reports how
    many first controls agree with the oracle's (the NLP is multi-modal from the cold start: DESIGN.md 6)."""
    import multiprocessing as mp
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import mpc_rl_for_avs_b200 as pkg
    cores = os.cpu_count() or 1
    n = max(cores * 2, int(seconds * cores / 0.08))      # ~0.08 s per oracle predict per core
    obs, rs, has = pkg.make_scenarios(n, M, seed=1234)
    obs, rs, has = obs.numpy(), rs.numpy(), has.numpy()
    items = [(obs[i], (rs[i] if has[i] else None)) for i in range(n)]
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        pool.map(_ref_one, items[:cores], chunksize=1)
        t0 = time.perf_counter()
        ref = pool.map(_ref_one, items, chunksize=1)
        dt = time.perf_counter() - t0
        out = {"value": n / dt, "unit": "solves/s", "cores": cores, "kind": "port",
               "sample": f"first {n} problems of the seed-1234 workload, one predict per task (SLSQP port of the NLP), {cores} processes, {dt:.1f} s"}
        if agent is not None:
            import numpy as np
            import torch
            ref = np.asarray(ref, dtype=np.float64)
            rsn = np.where(has.reshape(-1), rs.reshape(-1), np.nan).astype(np.float32)
            agent.reset()
            act, U = agent.predict_batch(torch.from_numpy(obs).cuda(agent.device), ref_speed=torch.from_numpy(rsn).cuda(agent.device),
                                         return_controls=True)
            torch.cuda.synchronize()
            act, U, status = act.cpu().numpy(), U.cpu().numpy(), agent.status[:n].cpu().numpy()
            cost64 = np.asarray(pool.map(_cost64, [(obs[i], (rs[i] if has[i] else None), U[i]) for i in range(n)], chunksize=8))
            du0 = np.abs(act.astype(np.float64) - ref[:, :2]).max(axis=1)
            below = cost64 <= ref[:, 2] * (1 + 1e-6) + 1e-6
            conv_idx = np.nonzero(status == 0)[0][:1024]          # bounded: about 5 s of host time
            confirmed = pool.map(_confirm, [(obs[i], (rs[i] if has[i] else None), U[i]) for i in conv_idx], chunksize=4)
            out["parity_sample"] = {"problems": n, "n_starts": agent.n_starts, "gpu_converged": int((status == 0).sum()),
                                    "gpu_settled": int(((status & ~32) == 0).sum()),
                                    "cost_at_or_below_cpu_port": int(below.sum()),
                                    "first_control_within_1e-3": int((du0 < 1e-3).sum()),
                                    "status0_checked": int(len(conv_idx)), "status0_confirmed_by_oracle": int(sum(confirmed)),
                                    "note": "against the SLSQP port timed here (one cold start; the golden fixtures of tests/ use the "
                                            "stronger best-of-portfolio oracle incl. the IPOPT-like interior point); the NLP is multi-modal"}
    return out


if __name__ == "__main__":
    main()
