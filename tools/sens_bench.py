"""Times the solution sensitivity (mpc_sensitivity) on the config-3 workload and reports its flags.

    python tools/sens_bench.py [--iters 20] [--warmup 3] [--out DIR]

make_scenarios(65536, 8, seed=1234), a 4-start predict_batch with controls, then sensitivity(U) at act_tol 1e-4 and
stat_tol 1e-3.  Launch time: CUDA events around each of `iters` sensitivity calls after `warmup` calls, against the
solve step (predict_batch, events around max(iters // 5, 3) steps).  Prints one JSON line: the card's name and power
limit (read in the same run), both times, their ratio, and the flag shares by solver status.  Writes nothing unless
--out is given."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mpc_rl_for_avs_b200 as pkg  # noqa: E402

CFG = {"horizon": 20, "weight_speed": 1.0, "weight_control": 1.0, "weight_input_diff": 1.0}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name()


def time_ms(fn, n):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sens_bench needs a CUDA device")
    B, M = a.batch, 8
    obs, rs, has = pkg.make_scenarios(B, M, seed=1234)
    obs = obs.cuda()
    rsn = torch.where(has.reshape(-1, 1), rs, torch.full_like(rs, float("nan"))).cuda()
    agent = pkg.BatchedPureMPC(CFG, vehicles_count=M + 1, max_batch=B, collision_check=True, weight_distance=10.0, n_starts=4)

    def solve():
        agent.reset()
        return agent.predict_batch(obs, rsn, return_controls=True)

    for _ in range(2):
        _, U = solve()
    torch.cuda.synchronize()
    status = agent.status[:B].cpu().numpy().copy()
    cost = agent.cost[:B].cpu().numpy().copy()
    sens = {}

    def run():
        sens.update(agent.sensitivity(U, act_tol=1e-4, stat_tol=1e-3))

    for _ in range(a.warmup):
        run()
    torch.cuda.synchronize()
    sens_ms = time_ms(run, a.iters)
    solve_ms = time_ms(solve, max(a.iters // 5, 3))
    # the solve above refilled the workspace with the same problems; differentiate the controls of the last solve
    _, U = solve()
    run()
    torch.cuda.synchronize()
    fl = sens["flags"].cpu().numpy()
    by_status = {}
    for s in np.unique(status):
        m = status == s
        by_status[int(s)] = dict(n=int(m.sum()), **{str(int(f)): float(np.mean(fl[m] == f)) for f in np.unique(fl[m])})
    out = {"metric": "sensitivity_ms", "card": card(), "batch": B, "n_starts": 4, "act_tol": 1e-4, "stat_tol": 1e-3,
           "sens_ms_median": float(np.median(sens_ms)), "sens_ms_min": float(np.min(sens_ms)),
           "sens_ms_max": float(np.max(sens_ms)), "solve_step_ms_median": float(np.median(solve_ms)),
           "ratio_to_solve": float(np.median(sens_ms) / np.median(solve_ms)),
           "ok_or_weak": float(np.mean((fl & ~2) == 0)), "flags_by_status": by_status}
    print(json.dumps(out), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "sens_bench.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
