"""Cost of a formation_hd_env target bank on the step path: the same workloads with and without a bank, timed with
CUDA events, alternating rounds in one process (so clock and co-tenant drift hit both arms alike).

    python scripts/bench_targets.py [--rounds 7] [--steps 200] [--out result.json]

Workloads (fp32, silent agents, auto-reset on):
  * fg_step_fused, random policy drawn and recorded in-kernel (bench.py's headline step): 131072 envs x 9 agents,
    episode_length = 25, so every 25th step resets every env;
  * step_bfs(3) at N = 9 (step kernel + controller kernel per step) and at N = 3 (one launch per step: the controller
    is compiled into the warp kernel).
The bank holds 7 tasks (random shapes and velocities); its index is -1 everywhere, so every reset draws its task.
Prints the card name and power limit with the numbers; the per-arm time is the median over rounds of the mean step
time of a round."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-formation_b200"))
from formation_gym.batched import BatchedFormationEnv  # noqa: E402

WORKLOADS = [("fg_step_fused 131072 x 9", 9, 131072, "step"), ("step_bfs(3) N=9", 9, 131072, "bfs"),
             ("step_bfs(3) N=3", 3, 1048576, "bfs")]


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info = "unknown"
    return name, info


def make(N, E, bank):
    kw = {}
    if bank:
        rng = np.random.default_rng(N)
        kw = dict(target_shapes=rng.uniform(-1, 1, (7, N, 2)), target_vels=rng.uniform(-1, 1, (7, 2)))
    env = BatchedFormationEnv("formation_hd_env", E, N, episode_length=25, seed=1, **kw)
    env.reset()
    return env


def run(env, how, steps):
    if how == "step":
        for _ in range(steps):
            env.step_random(record_actions=True)
    else:
        env.step_bfs(3, n_steps=steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_targets.py needs a CUDA device")
    name, info = card()
    print("device: %s; power.limit, clocks.max.sm: %s" % (name, info))
    res = {"device": name, "power_limit_and_max_sm_clock": info, "steps_per_round": a.steps, "rounds": a.rounds,
           "workloads": {}}
    for label, N, E, how in WORKLOADS:
        envs = {False: make(N, E, False), True: make(N, E, True)}
        for env in envs.values():                              # warm-up: modules, occupancy queries, clocks
            run(env, how, 50)
        torch.cuda.synchronize()
        times = {False: [], True: []}
        for r in range(a.rounds):
            for bank in ((False, True) if r % 2 == 0 else (True, False)):
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                run(envs[bank], how, a.steps)
                t1.record()
                t1.synchronize()
                times[bank].append(t0.elapsed_time(t1) * 1e3 / a.steps)
        med = {b: float(np.median(v)) for b, v in times.items()}
        spread = {b: float(np.max(v) - np.min(v)) for b, v in times.items()}
        res["workloads"][label] = {"envs": E, "agents": N, "us_per_step_no_bank": times[False],
                                   "us_per_step_bank": times[True], "median_no_bank": med[False],
                                   "median_bank": med[True], "ratio_bank_over_no_bank": med[True] / med[False]}
        print("%-26s no bank %8.2f us/step (spread %.2f)   bank %8.2f us/step (spread %.2f)   ratio %.4f"
              % (label, med[False], spread[False], med[True], spread[True], med[True] / med[False]))
        del envs
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
