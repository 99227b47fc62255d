"""Cost of the on-policy rollout buffer (formation_gym.rollout.StateRolloutBuffer) and of its GAE kernel (fg_gae),
timed with CUDA events, arms alternated round by round in one process (so clock and co-tenant drift hit every arm alike).

    python scripts/bench_rollout.py [--rounds 5] [--reps 20] [--out result.json]

Workloads (fp32, silent agents, auto-reset on, episode_length = 25): hd N = 9 x 131072 and hd N = 27 x 65536 at T = 25,
hd N = 9 x 65536 at T = 100, partial N = 4 x 262144 at T = 25.  Per workload, after one untimed rollout with
final_values (step_random(record_actions=True) + insert):
  * compute_returns: the buffer's call (one fg_gae launch) against the same recurrence written as a torch loop over t
    (where / mul / add / sub per step), us per call; and the k_gae kernel alone (torch.profiler, a separate phase after
    the timed rounds) with its algorithmic bytes -- reward, value, adv, ret once per (t, column), value[T], done once per
    (t, env) and final_value where done -- over the kernel time as a fraction of the HBM peak bench.py uses
    (MEASURED_PEAKS.json hbm_gbs, else its fallback);
  * a device-to-device copy_ that reads and writes half of k_gae's algorithmic bytes each (k_gae's own read / write
    mix), us per call: what a streaming kernel with that mix reaches on the card, next to k_gae's fraction;
  * insert: a rollout of T steps of step_random alone against start() + T x (step_random + insert), us per step;
  * one epoch of minibatches(n), n in {1, 4}: the buffer's (fg_obs_gather decode) against the same indexing of a stored
    obs [T,E,N,D] tensor (where it fits in free device memory), us per epoch;
  * bytes per env-step, computed from shapes, of this buffer, of an observation-level buffer, and of onpolicy's
    SharedReplayBuffer layout with share_obs.
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
from bench_replay import card, hbm_peak, timed  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402
from formation_gym.rollout import StateRolloutBuffer  # noqa: E402

EP = 25
GAMMA, LAM = 0.99, 0.95
WORKLOADS = [("hd N=9 x 131072, T=25", "formation_hd_env", 9, 131072, 25),
             ("hd N=27 x 65536, T=25", "formation_hd_env", 27, 65536, 25),
             ("hd N=9 x 65536, T=100", "formation_hd_env", 9, 65536, 100),
             ("partial N=4 x 262144, T=25", "formation_hd_partial_env", 4, 262144, 25)]
MINIBATCHES = (1, 4)


def torch_gae(buf, adv, ret):
    """The fg_gae recurrence as a torch loop over t (what a trainer writes without the kernel)."""
    d = buf.done[..., None]
    a = torch.zeros_like(buf.rewards[0])
    for t in range(buf.num_steps - 1, -1, -1):
        nv = torch.where(d[t], buf.final_values[t], buf.values[t + 1])
        delta = buf.rewards[t] + GAMMA * nv - buf.values[t]
        a = torch.where(d[t], delta, delta + (GAMMA * LAM) * a)
        adv[t] = a
        torch.add(a, buf.values[t], out=ret[t])


def obs_epoch(buf, obs_store, n, g):
    """One epoch over a stored obs [T,E,N,D] tensor, indexed like StateRolloutBuffer.minibatches."""
    T, E, N = buf.num_steps, buf.env.E, buf.env.N
    B = (T * E) // n
    perm = torch.randperm(T * E, device=obs_store.device, generator=g)
    flat = {"obs": obs_store.view(T * E, N, -1), "actions": buf.actions.view(T * E, N, -1),
            "log_probs": buf.log_probs.view(T * E, N), "values": buf.values[:T].reshape(T * E, N),
            "returns": buf.returns.view(T * E, N), "advantages": buf.advantages.view(T * E, N)}
    for i in range(n):
        rows = perm[i * B:(i + 1) * B]
        mb = {k: v[rows] for k, v in flat.items()}
        step = rows.div(E, rounding_mode="floor")
        mb["step_index"], mb["env_index"] = step, rows - step * E


def bytes_per_env_step(env):
    es = 4 if env.dtype == torch.float32 else 8
    N, A, D = env.N, env.act_dim, env.D
    rec = sum(es * (2 if k == "ideal_vel" else 2 * (env.L if k == "landmarks" else N)) for k in env.state_record_keys())
    # actions, log_probs, rewards, advantages, returns, values, final_values, done
    rest = es * N * A + 6 * es * N + 1
    # onpolicy SharedReplayBuffer (no RNN states / available actions): share_obs [N, N*D], obs [N, D], actions,
    # action_log_probs, rewards, value_preds, returns, advantages, masks, bad_masks, active_masks
    onpolicy = es * (N * N * D + N * D + N * A + 8 * N)
    return {"state_record_bytes": rec, "state_rollout": rec + rest, "observation_level": es * N * D + rest,
            "onpolicy_with_share_obs": onpolicy}


def kernel_time(fn, n, name):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    tot, cnt = 0.0, 0
    for e in prof.events():
        if e.device_type.name == "CUDA" and name in e.name:
            tot += e.device_time if hasattr(e, "device_time") else e.cuda_time
            cnt += 1
    return {"us_per_call": tot / n, "launches_per_call": cnt / n}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20, help="compute_returns calls per round and arm")
    ap.add_argument("--epochs", type=int, default=3, help="minibatch epochs per round and arm")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rollout.py needs a CUDA device")
    name, info = card()
    peak, peak_src = hbm_peak()
    print("device: %s; power.limit, clocks.max.sm: %s; HBM peak %.0f GB/s (%s)" % (name, info, peak, peak_src))
    res = {"device": name, "power_limit_and_max_sm_clock": info, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
           "episode_length": EP, "gamma": GAMMA, "gae_lambda": LAM, "rounds": a.rounds, "workloads": {}}
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    for label, scn, N, E, T in WORKLOADS:
        envs = {arm: BatchedFormationEnv(scn, E, N, episode_length=EP, seed=1) for arm in ("step", "step+insert")}
        for env in envs.values():
            env.reset()
        env = envs["step+insert"]
        dev = env.device
        g = torch.Generator(device=dev).manual_seed(0)
        buf = StateRolloutBuffer(env, T)
        lp = torch.randn(E, N, device=dev, generator=g)
        v = torch.randn(E, N, device=dev, generator=g)
        fv = torch.randn(E, N, device=dev, generator=g)

        def rollout(arm):
            e = envs[arm]
            if arm == "step":
                for _ in range(T):
                    e.step_random(record_actions=True)
                return
            buf.start()
            for _ in range(T):
                e.step_random(record_actions=True)
                buf.insert(e.actions, lp, v, final_values=fv)

        for arm in envs:                                     # warm-up: modules, allocations, clocks
            rollout(arm)
        nv = torch.randn(E, N, device=dev, generator=g)
        buf.compute_returns(nv, GAMMA, LAM)
        t_adv, t_ret = torch.empty_like(buf.advantages), torch.empty_like(buf.returns)
        torch_gae(buf, t_adv, t_ret)
        torch.cuda.synchronize()
        max_diff = max(float((t_adv - buf.advantages).abs().max()), float((t_ret - buf.returns).abs().max()))
        gae_fns = {"compute_returns": lambda: buf.compute_returns(nv, GAMMA, LAM),
                   "torch_loop": lambda: torch_gae(buf, t_adv, t_ret)}
        obs_store = None
        if torch.cuda.mem_get_info(dev)[0] > 2.5 * T * E * N * env.D * 4 + (4 << 30):
            obs_store = torch.randn(T, E, N, env.D, device=dev, generator=g)
        mb_fns = {}
        for n in MINIBATCHES:
            mb_fns[("state_minibatches", n)] = lambda n=n: [None for _ in buf.minibatches(n, generator=g)]
            if obs_store is not None:
                mb_fns[("obs_store_indexing", n)] = lambda n=n: obs_epoch(buf, obs_store, n, g)
        for f in list(gae_fns.values()) + list(mb_fns.values()):
            f()
        torch.cuda.synchronize()
        M = E * N
        n_done = int(buf.done.sum())
        alg = 16 * T * M + 4 * M + T * E + 4 * N * n_done     # fp32
        src = torch.empty(alg // 8, device=dev)
        dst = torch.empty_like(src)
        dst.copy_(src)
        t_copy = []
        t_gae = {k: [] for k in gae_fns}
        t_ins = {k: [] for k in envs}
        t_mb = {k: [] for k in mb_fns}
        for r in range(a.rounds):
            order = (lambda x: list(x)) if r % 2 == 0 else (lambda x: list(x)[::-1])
            for k in order(gae_fns):
                t_gae[k].append(timed(gae_fns[k], a.reps, ev))
            t_copy.append(timed(lambda: dst.copy_(src), a.reps, ev))
            for k in order(envs):
                t_ins[k].append(timed(lambda: rollout(k), 1, ev) / T)
            buf.compute_returns(nv, GAMMA, LAM)             # (the rollout arm cleared it)
            for k in order(mb_fns):
                t_mb[k].append(timed(mb_fns[k], a.epochs, ev))
        kt = kernel_time(gae_fns["compute_returns"], a.reps, "k_gae")
        bpe = bytes_per_env_step(env)
        med = lambda x: float(np.median(x))                 # noqa: E731
        out = {"envs": E, "agents": N, "scenario": scn, "num_steps": T, "columns": M, "dones_in_rollout": n_done,
               "bytes_per_env_step": bpe,
               "onpolicy_over_state_bytes": bpe["onpolicy_with_share_obs"] / bpe["state_rollout"],
               "rollout_bytes": {"state_rollout": bpe["state_rollout"] * T * E + 4 * M,
                                 "onpolicy_with_share_obs": bpe["onpolicy_with_share_obs"] * (T + 1) * E},
               "compute_returns": {k: {"us_per_call": t_gae[k], "median_us_per_call": med(t_gae[k])} for k in t_gae},
               "torch_loop_max_abs_diff": max_diff,
               "kernel_k_gae": dict(kt, algorithmic_bytes=alg,
                                    frac_of_hbm_peak=alg / (kt["us_per_call"] * 1e-6) / (peak * 1e9)),
               "copy_same_bytes": {"us_per_call": t_copy, "median_us_per_call": med(t_copy),
                                   "frac_of_hbm_peak": 8 * src.numel() / (med(t_copy) * 1e-6) / (peak * 1e9)},
               "insert": {k: {"us_per_step": t_ins[k], "median_us_per_step": med(t_ins[k])} for k in t_ins},
               "minibatch_epoch": {}}
        out["compute_returns"]["speedup_over_torch_loop"] = \
            out["compute_returns"]["torch_loop"]["median_us_per_call"] / \
            out["compute_returns"]["compute_returns"]["median_us_per_call"]
        out["insert"]["insert_us_per_step"] = out["insert"]["step+insert"]["median_us_per_step"] - \
            out["insert"]["step"]["median_us_per_step"]
        for (k, n), ts in t_mb.items():
            out["minibatch_epoch"].setdefault(str(n), {})[k] = {"us_per_epoch": ts, "median_us_per_epoch": med(ts)}
        if obs_store is None:
            out["minibatch_epoch"]["obs_store"] = "not measured: an obs [T,E,N,D] store does not fit beside the buffer"
        cr = out["compute_returns"]
        print("%-28s compute_returns %8.1f us (k_gae %.1f us, %.2f of HBM peak, %.0f MB; copy %.2f) vs torch loop"
              " %9.1f us (x%.1f) | insert +%.1f us/step | B/env-step state %d onpolicy %d (x%.0f)" % (
                  label, cr["compute_returns"]["median_us_per_call"], kt["us_per_call"],
                  out["kernel_k_gae"]["frac_of_hbm_peak"], alg / 1e6, out["copy_same_bytes"]["frac_of_hbm_peak"],
                  cr["torch_loop"]["median_us_per_call"], cr["speedup_over_torch_loop"], out["insert"]["insert_us_per_step"], bpe["state_rollout"],
                  bpe["onpolicy_with_share_obs"], out["onpolicy_over_state_bytes"]))
        for n in MINIBATCHES:
            row = out["minibatch_epoch"][str(n)]
            print("    minibatches(%d) epoch: state %9.1f us  obs store %s" % (
                n, row["state_minibatches"]["median_us_per_epoch"],
                "%9.1f us" % row["obs_store_indexing"]["median_us_per_epoch"] if "obs_store_indexing" in row else "-"))
        res["workloads"][label] = out
        del envs, env, buf, obs_store, gae_fns, mb_fns, t_adv, t_ret, src, dst
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
