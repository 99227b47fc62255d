"""Cost of the state-record replay buffer (formation_gym.replay.StateReplayBuffer) against an observation-level ring
holding the same transitions, timed with CUDA events, arms alternated round by round in one process (so clock and
co-tenant drift hit every arm alike).

    python scripts/bench_replay.py [--rounds 5] [--steps 20] [--capacity 8] [--out result.json]

Workloads (fp32, silent agents, auto-reset on, episode_length = 25): hd N = 9 x 131072, hd N = 27 x 65536,
partial N = 4 x 262144, hd N = 81 x 8192.  Per workload:
  * add: step_random(record_actions=True) alone, + StateReplayBuffer.add, + an observation-level ring's add (obs,
    next_obs = where(done, final_observation(), obs), act, reward, done), us per step;
  * sample(B), B in {4096, 65536}: StateReplayBuffer.sample against index_select over the observation ring, us per call;
  * decode: fg_obs_gather alone on 2B rows, and the bytes it writes over its kernel time as a fraction of the HBM peak
    bench.py uses (MEASURED_PEAKS.json hbm_gbs, else its fallback);
  * bytes per transition of both stores, computed from shapes.
Prints the card name and power limit with the numbers; a time is the median over rounds of a round's mean."""
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
from formation_gym.replay import StateReplayBuffer  # noqa: E402

EP = 25
FALLBACK_HBM_GBS = 6650.0                                    # bench.py's fallback when MEASURED_PEAKS.json is absent
WORKLOADS = [("hd N=9 x 131072", "formation_hd_env", 9, 131072), ("hd N=27 x 65536", "formation_hd_env", 27, 65536),
             ("partial N=4 x 262144", "formation_hd_partial_env", 4, 262144), ("hd N=81 x 8192", "formation_hd_env", 81, 8192)]
ADD_ARMS = ("step", "step+state_add", "step+obs_add")
BATCHES = (4096, 65536)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info = "unknown"
    return name, info


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback of bench.py"


class ObsRing:
    """The observation-level store a MADDPG trainer keeps: obs, next_obs, act, reward, done per transition."""

    def __init__(self, env, T):
        kw = dict(device=env.device, dtype=env.dtype)
        self.env, self.T, self.j, self.n = env, T, 0, 0
        self.obs = torch.zeros(T, env.E, env.N, env.D, **kw)
        self.next_obs = torch.zeros(T, env.E, env.N, env.D, **kw)
        self.act = torch.zeros(T, env.E, env.N, env.act_dim, **kw)
        self.rew = torch.zeros(T, env.E, env.N, **kw)
        self.done = torch.zeros(T, env.E, dtype=torch.bool, device=env.device)
        self.prev = env.obs.clone()

    def add(self, actions):
        env, j = self.env, self.j
        self.obs[j].copy_(self.prev)
        d = env.done[:, 0]
        torch.where(d[:, None, None], env.final_observation(), env.obs, out=self.next_obs[j])
        self.act[j].copy_(actions)
        self.rew[j].copy_(env.reward[..., 0])
        self.done[j].copy_(d)
        self.prev.copy_(env.obs)
        self.j, self.n = (j + 1) % self.T, min(self.n + 1, self.T)

    def sample(self, B, generator=None):
        E = self.env.E
        k = torch.randint(0, self.n * E, (B,), device=self.env.device, generator=generator)
        out = {}
        for name in ("obs", "next_obs", "act", "rew", "done"):
            t = getattr(self, name)
            out[name] = t.view(self.T * E, *t.shape[2:]).index_select(0, k)
        return out


def bytes_per_transition(env):
    es = 4 if env.dtype == torch.float32 else 8
    N, A = env.N, env.act_dim
    rest = es * N * A + es * N + 1                          # act, reward, done
    rec = sum(es * (2 if k == "ideal_vel" else 2 * (env.L if k == "landmarks" else N)) for k in env.state_record_keys())
    return {"state_record_bytes": rec, "state_level": 2 * rec + rest, "observation_level": 2 * es * N * env.D + rest}


def timed(fn, n, ev):
    ev[0].record()
    for _ in range(n):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) * 1e3 / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20, help="steps per round and add arm")
    ap.add_argument("--capacity", type=int, default=8)
    ap.add_argument("--samples", type=int, default=20, help="sample calls per round and arm")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_replay.py needs a CUDA device")
    name, info = card()
    peak, peak_src = hbm_peak()
    print("device: %s; power.limit, clocks.max.sm: %s; HBM peak %.0f GB/s (%s)" % (name, info, peak, peak_src))
    res = {"device": name, "power_limit_and_max_sm_clock": info, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
           "episode_length": EP, "capacity": a.capacity, "rounds": a.rounds, "workloads": {}}
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    for label, scn, N, E in WORKLOADS:
        envs = {arm: BatchedFormationEnv(scn, E, N, episode_length=EP, seed=1, record_final=True) for arm in ADD_ARMS}
        for env in envs.values():
            env.reset()
        sbuf = StateReplayBuffer(envs["step+state_add"], a.capacity)
        sbuf.mark_start()
        oring = ObsRing(envs["step+obs_add"], a.capacity)
        adds = {"step": lambda env: None, "step+state_add": lambda env: sbuf.add(env.actions),
                "step+obs_add": lambda env: oring.add(env.actions)}

        def one(arm):
            env = envs[arm]
            env.step_random(record_actions=True)
            adds[arm](env)

        for arm in ADD_ARMS:                                  # warm-up: fills both rings, modules, clocks
            for _ in range(a.capacity + 1):
                one(arm)
        torch.cuda.synchronize()
        t_add = {arm: [] for arm in ADD_ARMS}
        g = torch.Generator(device=envs["step"].device).manual_seed(0)
        s_arms = ["state_sample", "obs_sample", "decode"]
        t_smp = {(arm, B): [] for arm in s_arms for B in BATCHES}
        rows = {B: torch.randint(0, sbuf.num_records // 2, (2 * B,), device=envs["step"].device, generator=g)
                for B in BATCHES}
        env_s = envs["step+state_add"]
        fns = {"state_sample": lambda B: sbuf.sample(B, generator=g), "obs_sample": lambda B: oring.sample(B, generator=g),
               "decode": lambda B: env_s.gather_observations(sbuf.states, rows[B])}
        for B in BATCHES:
            for arm in s_arms:
                fns[arm](B)
        for r in range(a.rounds):
            for arm in (ADD_ARMS if r % 2 == 0 else ADD_ARMS[::-1]):
                t_add[arm].append(timed(lambda: one(arm), a.steps, ev))
            for B in BATCHES:
                for arm in (s_arms if r % 2 == 0 else s_arms[::-1]):
                    t_smp[(arm, B)].append(timed(lambda: fns[arm](B), a.samples, ev))
        env = envs["step"]
        bpt = bytes_per_transition(env)
        out = {"envs": E, "agents": N, "scenario": scn, "bytes_per_transition": bpt,
               "ratio_observation_over_state_bytes": bpt["observation_level"] / bpt["state_level"], "add": {}, "sample": {}}
        es = 4
        for arm in ADD_ARMS:
            out["add"][arm] = {"us_per_step": t_add[arm], "median_us_per_step": float(np.median(t_add[arm]))}
        base = out["add"]["step"]["median_us_per_step"]
        line = "%-22s B/transition state %6d obs %8d (x%.1f) | step %8.1f us" % (
            label, bpt["state_level"], bpt["observation_level"], out["ratio_observation_over_state_bytes"], base)
        for arm in ADD_ARMS[1:]:
            m = out["add"][arm]["median_us_per_step"]
            out["add"][arm]["add_us_per_step"] = m - base
            line += "  %s +%.1f us" % (arm.split("+")[1], m - base)
        print(line)
        for B in BATCHES:
            row = {arm: {"us_per_call": t_smp[(arm, B)], "median_us_per_call": float(np.median(t_smp[(arm, B)]))}
                   for arm in s_arms}
            wr = 2 * B * N * env.D * es                        # bytes the decode writes (obs + next_obs)
            row["decode"]["bytes_written"] = wr
            row["decode"]["frac_of_hbm_peak_written"] = wr / (row["decode"]["median_us_per_call"] * 1e-6) / (peak * 1e9)
            out["sample"][str(B)] = row
            print("    B=%-6d state sample %8.1f us  obs-ring sample %8.1f us  decode %8.1f us = %.2f of HBM peak" % (
                B, row["state_sample"]["median_us_per_call"], row["obs_sample"]["median_us_per_call"],
                row["decode"]["median_us_per_call"], row["decode"]["frac_of_hbm_peak_written"]))
        res["workloads"][label] = out
        del envs, sbuf, oring, fns, adds, env, env_s
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
