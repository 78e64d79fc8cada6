"""Fixed 4 vs fixed 8 vs adaptive 4 -> 8 starts on the config-3 workload, timed alternately in one process.

    python tools/adaptive_starts_bench.py [--steps 20] [--warmup 5] [--rounds 3] [--rel-gap 1e-3]

Workload exactly as bench.py builds config 3: 65536 problems per step from make_scenarios(65536, 8, seed=1234 + 1000 s),
eight rotating batches (8 x 19.4 MB of inputs > the 126 MB L2), distance cost 10, collision check on, the RL reference
speed on half of the batch.  Each round times every arm over `--steps` steps (CUDA events around the steps, and the
library's own events around every solve launch, `timing_begin/end`); the arms alternate within a round so that they
share the machine's conditions.  Per arm: median ms per step over the rounds with its min / max, problems/s, solves/s,
kernel ms.  Then one untimed pass over the eight batches gives mean iterations per problem, the extended fraction and
the mean starts run per problem.  `tail_ms` of the adaptive arm is its kernel time minus the time the same solves would
take at the fixed arms' rate (kernel_4 + (kernel_8 - kernel_4) x extended fraction): what publishing the extra starts
only when a problem's last base start ends adds to the launch.  Prints one JSON line, with the GPU's name and power
limit read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

H, M, W_DIST, B = 20, 8, 10.0, 65536
CFG = {"horizon": H, "weight_speed": 1.0, "weight_control": 1.0, "weight_input_diff": 1.0}


def gpu_info(index: int) -> dict:
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit": q[1], "max_sm_clock": q[2]}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--rel-gap", type=float, default=1e-3)
    ap.add_argument("--max-starts", type=int, default=8)
    args = ap.parse_args()
    if args.steps < 20:
        ap.error("--steps must be at least 20")

    import torch
    import mpc_rl_for_avs_b200 as pkg
    if not torch.cuda.is_available():
        raise SystemExit("adaptive_starts_bench.py needs a CUDA device: the MPC path has no CPU implementation")
    dev = torch.device("cuda", 0)
    batches = []
    for s in range(8):
        obs, rs, has = pkg.make_scenarios(B, M, seed=1234 + 1000 * s)
        rsn = torch.where(has.reshape(-1, 1), rs, torch.full_like(rs, float("nan"))).reshape(-1).contiguous()
        batches.append((obs.contiguous().to(dev), rsn.to(dev)))

    def agent(n_starts, adaptive=False):
        a = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=B, device=0, collision_check=True, weight_distance=W_DIST,
                               n_starts=n_starts)
        if adaptive:
            a.set_adaptive_starts(args.max_starts, args.rel_gap)
        return a

    arms = {"fixed_4": agent(4), f"fixed_{args.max_starts}": agent(args.max_starts), "adaptive": agent(4, adaptive=True)}

    def step(a, i):
        o, r = batches[i % len(batches)]
        a.reset()
        a.predict_batch(o, ref_speed=r)

    for a in arms.values():
        for i in range(args.warmup):
            step(a, i)
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    kern = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, a in arms.items():
            a.timing_begin()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                step(a, i)
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.steps)
            kern[k].append(a.timing_end()["solve_ms"])

    out = {"metric": "adaptive_starts_config3", "problems_per_step": B, "steps": args.steps, "rounds": args.rounds,
           "rel_gap": args.rel_gap, "max_starts": args.max_starts, "gpu": gpu_info(0), "arms": {}}
    for k, a in arms.items():
        its, ext = [], []
        for i in range(len(batches)):
            step(a, i)
            torch.cuda.synchronize()
            its.append(float(a.iters[:B].float().mean()))
            if a.max_starts:
                ext.append(float(a.extended[:B].float().mean()))
        med = statistics.median(ms[k])
        starts = 4 + (args.max_starts - 4) * statistics.mean(ext) if ext else a.n_starts
        out["arms"][k] = {"ms_per_step": med, "ms_min": min(ms[k]), "ms_max": max(ms[k]), "problems_per_s": B / (med * 1e-3),
                          "solves_per_s": B * starts / (med * 1e-3), "kernel_ms": statistics.median(kern[k]),
                          "mean_iters": statistics.mean(its), "mean_starts": starts}
        if ext:
            out["arms"][k]["extended_fraction"] = statistics.mean(ext)
    k4, k8, ka = (out["arms"][k]["kernel_ms"] for k in ("fixed_4", f"fixed_{args.max_starts}", "adaptive"))
    f = out["arms"]["adaptive"]["extended_fraction"]
    out["arms"]["adaptive"]["tail_ms"] = ka - (k4 + (k8 - k4) * f)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
