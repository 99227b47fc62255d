"""Cost of terminal blocks (record_final) on the step path: the same workloads with and without a block, timed per step
with CUDA events, alternating arms round by round in one process (so clock and co-tenant drift hit every arm alike).

    python scripts/bench_final.py [--rounds 5] [--episodes 2] [--out result.json]

Arms (fp32, silent agents, auto-reset on, episode_length = 25, so every 25th step ends every episode):
  * plain:     step_random(record_actions=True) without a block;
  * final:     the same step with record_final=True (the extension instantiation of the step kernel);
  * final+obs: the same step followed by final_observation() on every step, as a CUDA-graph trainer would call it.
Each arm's step times are split into the steps that end the episodes and the others.  Prints the card name and power
limit with the numbers; an arm's time is the median over rounds of the mean step time of a round."""
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

EP = 25
WORKLOADS = [("hd N=9 x 131072", "formation_hd_env", 9, 131072), ("hd N=27 x 65536", "formation_hd_env", 27, 65536),
             ("basic N=3 x 1M", "basic_formation_env", 3, 1 << 20),
             ("partial N=4 x 262144", "formation_hd_partial_env", 4, 262144),
             ("obs_env N=4 x 262144", "formation_hd_obs_env", 4, 262144), ("hd N=81 x 8192", "formation_hd_env", 81, 8192)]
ARMS = ("plain", "final", "final+obs")


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info = "unknown"
    return name, info


def make(scn, N, E, arm):
    env = BatchedFormationEnv(scn, E, N, episode_length=EP, seed=1, record_final=(arm != "plain"))
    env.reset()
    return env


def run(env, arm, steps, ev):
    """`steps` steps; ev[s] = (start, end) events around step s (and its final_observation)."""
    for s in range(steps):
        ev[s][0].record()
        env.step_random(record_actions=True)
        if arm == "final+obs":
            env.final_observation()
        ev[s][1].record()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=2, help="episodes per round (every env ends one each 25 steps)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_final.py needs a CUDA device")
    name, info = card()
    print("device: %s; power.limit, clocks.max.sm: %s" % (name, info))
    steps = EP * a.episodes
    res = {"device": name, "power_limit_and_max_sm_clock": info, "episode_length": EP, "steps_per_round": steps,
           "rounds": a.rounds, "workloads": {}}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for label, scn, N, E in WORKLOADS:
        envs = {arm: make(scn, N, E, arm) for arm in ARMS}
        for arm, env in envs.items():                          # warm-up: modules, occupancy queries, clocks
            run(env, arm, EP, ev)
        torch.cuda.synchronize()
        t_end = {arm: [] for arm in ARMS}
        t_mid = {arm: [] for arm in ARMS}
        for r in range(a.rounds):
            order = ARMS if r % 2 == 0 else ARMS[::-1]
            for arm in order:
                env = envs[arm]
                phase = env._tick                              # host tick = steps since the reset (one per step)
                run(env, arm, steps, ev)
                torch.cuda.synchronize()
                t = np.array([e0.elapsed_time(e1) * 1e3 for e0, e1 in ev])
                # the step taken with host tick k is the (k mod EP)-th of its episode (reset took tick 0)
                ends = np.array([((phase + s) % EP) == 0 for s in range(steps)])
                t_end[arm].append(float(t[ends].mean()))
                t_mid[arm].append(float(t[~ends].mean()))
        out = {"envs": E, "agents": N, "scenario": scn}
        line = "%-22s" % label
        for arm in ARMS:
            me, mm = float(np.median(t_end[arm])), float(np.median(t_mid[arm]))
            mean = (me + (EP - 1) * mm) / EP
            out[arm] = {"us_ending_step": t_end[arm], "us_other_step": t_mid[arm], "median_ending_step": me,
                        "median_other_step": mm, "amortised_us_per_step": mean}
            line += "  %s: end %7.2f other %7.2f amort %7.2f" % (arm, me, mm, mean)
        base = out["plain"]["amortised_us_per_step"]
        for arm in ARMS[1:]:
            out[arm]["ratio_amortised_over_plain"] = out[arm]["amortised_us_per_step"] / base
        print(line + "   (us/step)")
        res["workloads"][label] = out
        del envs
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
