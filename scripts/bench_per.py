"""Cost of prioritized replay (formation_gym.replay.PrioritizedStateReplayBuffer) next to the uniform
StateReplayBuffer, timed with CUDA events, arms alternated round by round in one process (so clock and co-tenant drift
hit every arm alike).

    python scripts/bench_per.py [--rounds 5] [--steps 20] [--samples 20] [--out result.json]

Workloads (fp32, silent agents, auto-reset on, episode_length = 25): those of scripts/bench_replay.py at capacity 8 --
hd N = 9 x 131072, hd N = 27 x 65536, partial N = 4 x 262144, hd N = 81 x 8192 -- and hd N = 9 x 65536 at capacity 100
(M = 6.5 M leaves, tree depth 5).  Per workload:
  * add: step_random(record_actions=True) alone, + StateReplayBuffer.add, + PrioritizedStateReplayBuffer.add, us per
    step; the PER extra is the difference of the two add arms;
  * sample(B), B in {4096, 65536}, for both buffers, and update_priorities(B), us per call.  Every timed update gets a
    batch sampled (untimed) after the last add(), so its entries are live -- a batch from before an add() whose slot
    was overwritten is skipped by the stamp check and would time the skip path; `live_fraction` records the share of
    update entries whose slot stamp still matched and whose leaf was > 0 when the batches were drawn;
  * kernel times (torch.profiler, a separate phase after the timed rounds): k_per_sample per sample call, and the sum of
    the update's kernels (k_per_claim, k_per_write, one k_per_level per tree level) per update call.
Prints the card name and power limit with the numbers; a time is the median over rounds of a round's mean."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-formation_b200"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from bench_replay import card, timed  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402
from formation_gym.replay import PrioritizedStateReplayBuffer, StateReplayBuffer  # noqa: E402

EP = 25
WORKLOADS = [("hd N=9 x 131072", "formation_hd_env", 9, 131072, 8), ("hd N=27 x 65536", "formation_hd_env", 27, 65536, 8),
             ("partial N=4 x 262144", "formation_hd_partial_env", 4, 262144, 8),
             ("hd N=81 x 8192", "formation_hd_env", 81, 8192, 8), ("hd N=9 x 65536, T=100", "formation_hd_env", 9, 65536, 100)]
ADD_ARMS = ("step", "step+uniform_add", "step+per_add")
BATCHES = (4096, 65536)


def kernel_times(fns, n):
    """Device time per call of the fg_per kernels, from a torch.profiler trace of n calls of each fn."""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name, (fn, kernels) in fns.items():
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                fn()
            torch.cuda.synchronize()
        tot, cnt = 0.0, 0
        for e in prof.events():
            if e.device_type.name == "CUDA" and any(k in e.name for k in kernels):
                tot += e.device_time if hasattr(e, "device_time") else e.cuda_time
                cnt += 1
        out[name] = {"us_per_call": tot / n, "kernel_launches_per_call": cnt / n}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20, help="steps per round and add arm")
    ap.add_argument("--samples", type=int, default=20, help="sample / update calls per round and arm")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_per.py needs a CUDA device")
    name, info = card()
    print("device: %s; power.limit, clocks.max.sm: %s" % (name, info))
    res = {"device": name, "power_limit_and_max_sm_clock": info, "episode_length": EP, "rounds": a.rounds,
           "workloads": {}}
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    for label, scn, N, E, T in WORKLOADS:
        envs = {arm: BatchedFormationEnv(scn, E, N, episode_length=EP, seed=1, record_final=True) for arm in ADD_ARMS}
        for env in envs.values():
            env.reset()
        ubuf = StateReplayBuffer(envs["step+uniform_add"], T)
        pbuf = PrioritizedStateReplayBuffer(envs["step+per_add"], T)
        ubuf.mark_start()
        pbuf.mark_start()
        adds = {"step": lambda env: None, "step+uniform_add": lambda env: ubuf.add(env.actions),
                "step+per_add": lambda env: pbuf.add(env.actions)}

        def one(arm):
            env = envs[arm]
            env.step_random(record_actions=True)
            adds[arm](env)

        for arm in ADD_ARMS:                                  # warm-up: fills both rings, modules, clocks
            for _ in range(T + 1):
                one(arm)
        dev = envs["step"].device
        g = torch.Generator(device=dev).manual_seed(0)
        tds = {B: torch.randn(B, device=dev, generator=g) for B in BATCHES}
        pending, live = {B: [] for B in BATCHES}, {B: [] for B in BATCHES}

        def refill(B, n):
            """n fresh batches for the next n updates (untimed; nothing is added before they are used)."""
            pending[B] = []
            for _ in range(n):
                b = pbuf.sample(B, generator=g)
                for k in ("obs", "next_obs", "actions", "reward"):   # an update reads index / stamp only
                    del b[k]
                pending[B].append(b)
            for b in pending[B]:
                ok = (pbuf._stamp_dev[b["slot"]] == b["stamp"]) & (pbuf._leaf[b["index"]] > 0)
                live[B].append(float(ok.double().mean()))
            torch.cuda.synchronize()

        fns = {"uniform_sample": lambda B: ubuf.sample(B, generator=g),
               "per_sample": lambda B: pbuf.sample(B, 0.4, generator=g),
               "per_update": lambda B: pbuf.update_priorities(pending[B].pop(), tds[B])}
        for B in BATCHES:
            refill(B, 1)
            for f in fns.values():
                f(B)
        torch.cuda.synchronize()
        t_add = {arm: [] for arm in ADD_ARMS}
        t_smp = {(arm, B): [] for arm in fns for B in BATCHES}
        for r in range(a.rounds):
            for arm in (ADD_ARMS if r % 2 == 0 else ADD_ARMS[::-1]):
                t_add[arm].append(timed(lambda: one(arm), a.steps, ev))
            for B in BATCHES:
                refill(B, a.samples)
                for arm in (list(fns) if r % 2 == 0 else list(fns)[::-1]):
                    t_smp[(arm, B)].append(timed(lambda: fns[arm](B), a.samples, ev))
        out = {"envs": E, "agents": N, "scenario": scn, "capacity": T, "leaves": T * E, "tree_depth": pbuf.depth,
               "tree_bytes": 8 * (pbuf._leaf.numel() + pbuf._sum.numel() + pbuf._min.numel()),
               "scratch_bytes": 4 * pbuf._scratch.numel(), "add": {}, "calls": {}}
        for arm in ADD_ARMS:
            out["add"][arm] = {"us_per_step": t_add[arm], "median_us_per_step": float(np.median(t_add[arm]))}
        med = {arm: out["add"][arm]["median_us_per_step"] for arm in ADD_ARMS}
        out["add"]["uniform_add_us"] = med["step+uniform_add"] - med["step"]
        out["add"]["per_add_us"] = med["step+per_add"] - med["step"]
        out["add"]["per_extra_over_uniform_us"] = med["step+per_add"] - med["step+uniform_add"]
        print("%-24s depth %d | step %8.1f us  uniform add +%.1f us  PER add +%.1f us (extra %+.1f us)" % (
            label, pbuf.depth, med["step"], out["add"]["uniform_add_us"], out["add"]["per_add_us"],
            out["add"]["per_extra_over_uniform_us"]))
        for B in BATCHES:
            refill(B, a.samples + 1)
        kt = kernel_times({"fg_per_sample B=%d" % B: (lambda B=B: fns["per_sample"](B), ("k_per_sample",))
                           for B in BATCHES} |
                          {"fg_per_update B=%d" % B: (lambda B=B: fns["per_update"](B),
                                                      ("k_per_claim", "k_per_write", "k_per_level")) for B in BATCHES},
                          a.samples)
        for B in BATCHES:
            row = {arm: {"us_per_call": t_smp[(arm, B)], "median_us_per_call": float(np.median(t_smp[(arm, B)]))}
                   for arm in fns}
            row["kernel_fg_per_sample"] = kt["fg_per_sample B=%d" % B]
            row["kernels_fg_per_update"] = kt["fg_per_update B=%d" % B]
            row["per_update"]["live_fraction"] = {"min": min(live[B]), "mean": float(np.mean(live[B]))}
            row["per_sample_at_or_below_uniform"] = \
                row["per_sample"]["median_us_per_call"] <= row["uniform_sample"]["median_us_per_call"]
            out["calls"][str(B)] = row
            print("    B=%-6d sample uniform %8.1f us  PER %8.1f us (kernel %.1f us) | update %8.1f us (kernels %.1f us,"
                  " %.0f launches, live %.3f)" % (B, row["uniform_sample"]["median_us_per_call"],
                                       row["per_sample"]["median_us_per_call"], row["kernel_fg_per_sample"]["us_per_call"],
                                       row["per_update"]["median_us_per_call"], row["kernels_fg_per_update"]["us_per_call"],
                                       row["kernels_fg_per_update"]["kernel_launches_per_call"], min(live[B])))
        res["workloads"][label] = out
        del envs, ubuf, pbuf, fns, adds, pending, tds
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
