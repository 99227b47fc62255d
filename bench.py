#!/usr/bin/env python
"""bench.py -- agent-steps/sec of the gym-formation MPE step path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] --steps K --warmup W   # CPU reference arm

One "step" = one env step (MultiAgentEnv.step semantics) of EVERY env of the batch under the random policy
(act ~ U(-1,1), test.py:20): ONE launch of the fused step kernel (fg_step_fused with random_actions = 2: the
actions are drawn from Philox inside the kernel AND recorded in the action buffer, then _set_action + World.step +
observation + reward + done + auto-reset).  `--two-kernels` runs the round-1 form instead (fg_random_actions
kernel, then fg_step_fused reading the action buffer); both give bit-identical results.  Workload
(config.workload): formation_hd_env, 9 agents, 131072 envs per GPU (= the north star's 1M envs on
8 GPUs), episode_length 25, fp32.  A step moves 131072 * 2437 B = 319 MB > the 126 MB L2, so
every timed iteration streams from/to HBM (no L2 flush needed).

Printed JSON keys beyond the base contract: `roofline` (fused step kernel vs measured HBM peak),
`cpu_baseline` (the UNMODIFIED reference, staged by oracle/make_ref.py into oracle/_ref, on the host
cores; N=1 only; the loop port's figure beside it), `e2e` (same metric through the public API with
pinned HOST buffers: H2D of the actions and D2H of obs/reward/done inside the timed region),
`clocks`, `gpu_launches`, `strong_scaling` (BASELINE configs[2] / configs[3] split evenly over the
ranks), `state_hash` (64-bit checksum of a fixed job's final state, identical at 1/2/4/8 ranks),
`also` (N=1 only: configs[0], configs[1], the configs[4] env-count sweep, u_noise run, ...).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, "gym-formation_b200"), ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "agent-steps/sec (formation_hd_env, random policy)"
UNIT = "agent-steps/s"
FALLBACK_HBM_GBS = 6650.0          # /opt/skills/guides/B200_PROFILING.md fallback


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=25)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scenario", default="formation_hd_env")
    ap.add_argument("--agents", type=int, default=9)
    ap.add_argument("--envs-per-gpu", type=int, default=131072)
    ap.add_argument("--episode-length", type=int, default=25)
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-obs", action="store_true", help="state+reward only (B_state accounting)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = max(10, min(--steps, 100))")
    ap.add_argument("--graph-steps", type=int, default=50,
                    help="env steps per CUDA graph in the timed region (0 = plain per-step launches)")
    ap.add_argument("--cpu-seconds", type=float, default=3.0)
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling lines and the state hash")
    ap.add_argument("--two-kernels", action="store_true",
                    help="random-policy kernel + step kernel per step instead of the policy fused into the step kernel")
    ap.add_argument("--u-noise", type=float, default=0.0, help="motor noise of the headline workload (core.py:232-236)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (obs, reward, done, individual reward, "
                         "recorded actions) as DIR/<name>.npy, for a fixed sample of envs when all would exceed 16 MB")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    return a


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "samples": len(sm),
                "reasons": sorted(reasons)}


def reference_cli(scenario, N, procs=0, seconds=None, max_steps=None, episode_length=25, warmup=None, timeout=900):
    """Run the UNMODIFIED reference (oracle/ref_harness.py: /root/reference here, the byte-for-byte staged copy
    oracle/_ref on the GPU box) in a clean subprocess -- its package is also called `formation_gym` -- one env per
    process like the reference's SubprocVecEnv.  Returns the harness' JSON dict or None when no tree is there."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_harness.py"), "--scenario", scenario, "--agents", str(N),
           "--procs", str(procs), "--episode-length", str(episode_length)]
    cmd += ["--seconds", str(seconds if seconds is not None else 1e9)]
    if max_steps is not None:
        cmd += ["--max-steps", str(max_steps)]
    if warmup is not None:
        cmd += ["--warmup", str(warmup)]
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
        d = json.loads(line)
        return None if "unavailable" in d else d
    except Exception:
        return None


def run_reference(a):
    """CPU reference arm: the reference's OWN implementation of the path -- the unmodified files
    formation_gym/{__init__,core,environment,scenario}.py + envs/ (staged by oracle/make_ref.py), driven through
    make_env(...).step() with the random policy -- on all host cores, one env per process like the reference's
    SubprocVecEnv (train/maddpg-v2/utils/env_wrappers.py:48-55).  A 'step' = one env step of that batch of P envs.
    Falls back to the loop port (oracle/ref_loop_port.py) only when no reference tree is available."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    N, K, W = a.agents, a.steps, a.warmup
    # keep the whole run within a few minutes whatever K is
    per_step = {3: 0.006, 9: 0.02, 27: 0.08, 243: 3.5}.get(N, 0.0002 * N * N + 0.002 * N)
    K_eff = max(1, min(K, int(120.0 / per_step)))
    Wn = min(W, 10)
    r = reference_cli(a.scenario, N, procs, None, K_eff, a.episode_length, Wn)
    if r is not None:
        kind, value, wall = "reference", r["agent_steps_per_s"], r["wall_s"]
        sample = ("%d envs (one per host core, %d processes) x %d env-steps of %s N=%d, episode_length %d; the UNMODIFIED "
                  "reference (formation_gym.make_env(...).step, files staged from %s; numpy %s, scipy %s)"
                  % (procs, procs, K_eff, a.scenario, N, a.episode_length,
                     "oracle/_ref" if r["reference_root"].endswith("_ref") else r["reference_root"], r["numpy"], r["scipy"]))
    else:
        import multiprocessing as mp
        import numpy as np
        from oracle import ref_loop_port as rp

        def worker(q, seed):
            np.random.seed(seed)
            env = rp.RefLoopEnv(a.scenario, N, a.episode_length)
            acts = lambda: [np.random.uniform(-1, 1, 2) for _ in range(N)]  # noqa: E731
            for _ in range(Wn):
                env.step(acts())
            t0 = time.perf_counter()
            for _ in range(K_eff):
                _, _, done_n, _ = env.step(acts())
                if all(done_n):
                    env.reset()
            q.put(time.perf_counter() - t0)

        ctx = mp.get_context("fork")
        q = ctx.Queue()
        ps = [ctx.Process(target=worker, args=(q, 100 + k)) for k in range(procs)]
        for p in ps:
            p.start()
        times = [q.get() for _ in ps]
        for p in ps:
            p.join()
        wall = max(times)
        kind, value = "port", procs * N * K_eff / wall
        sample = ("%d envs (one per host core, %d processes) x %d env-steps of %s N=%d, episode_length %d; "
                  "per-env Python/numpy loop port of the reference (oracle/ref_loop_port.py, scipy "
                  "directed_hausdorff=%s) -- no reference tree available" % (procs, procs, K_eff, a.scenario, N,
                                                                          a.episode_length, rp.HAVE_SCIPY))
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": K_eff, "warmup": Wn, "ms_per_step": wall / K_eff * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(a, procs, "cpu"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def workload_config(a, envs_per_unit, where):
    return {"workload": "%s N=%d, %d envs per %s, episode_length %d, random policy U(-1,1), auto-reset"
                        % (a.scenario, a.agents, envs_per_unit, "GPU" if where == "gpu" else "run",
                           a.episode_length),
            "scenario": a.scenario, "agents": a.agents, "envs_per_gpu": envs_per_unit if where == "gpu" else None,
            "episode_length": a.episode_length, "obs": not a.no_obs,
            "launch": (("cuda graph of per-step launches" if a.graph_steps > 0 else "per-step launches") +
                       ("; random-policy kernel + fused step kernel per step" if a.two_kernels else
                        "; one kernel per step (random policy drawn and recorded inside the fused step kernel)"))
            if where == "gpu" else None,
            "l2": "inputs larger than L2 (step traffic > 126 MB), no flush" if where == "gpu" else None}


DUMP_BYTES = 16 * 10 ** 6


def env_snapshot(torch, env):
    """Host Philox tick and a copy of every device buffer of a BatchedFormationEnv (state, outputs, device tick)."""
    return env._tick, {k: v.clone() for k, v in vars(env).items() if torch.is_tensor(v) and v.is_cuda}


def env_restore(env, snapshot):
    """Put a snapshot back in place: the env's buffers keep their addresses, so captured CUDA graphs stay valid."""
    env._tick = snapshot[0]
    for k, v in snapshot[1].items():
        getattr(env, k).copy_(v)


def dump_outputs(out_dir, torch, env):
    """What the step last returned -- obs, reward, done, individual reward -- and the actions it recorded, as
    DIR/<name>.npy in the env's float type.  Envs are sampled with a fixed seed (ascending index order) when all of
    them would exceed DUMP_BYTES."""
    import numpy as np
    outs = {"obs": env.obs, "reward": env.reward, "done": env.done, "individual_reward": env.indiv,
            "actions": env.actions}
    outs = {k: v for k, v in outs.items() if v is not None}
    per_env = sum(v[0].numel() for v in outs.values()) * torch.finfo(env.dtype).bits // 8
    n = max(1, min(env.E, DUMP_BYTES // per_env))
    idx = np.sort(np.random.RandomState(0).choice(env.E, n, replace=False)) if n < env.E else np.arange(env.E)
    sel = torch.as_tensor(idx, device=env.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in outs.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.index_select(0, sel).to(env.dtype).cpu().numpy())


def run_b200(a):
    import torch
    import torch.distributed as dist
    import formation_gym
    from formation_gym import distributed as fgd

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the step path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    cpus = fgd.bind_to_gpu(local_rank)            # NUMA-local cores before any pinned allocation (no-op on 1-node hosts)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL writes its version banner / debug lines to stdout: send them to a file so that stdout carries
        # exactly ONE JSON line whatever NCCL_DEBUG level the launcher chose
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/fg_bench_nccl.%h.%p.log")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"          # NCCL honours the debug file only above the VERSION level
        dist.init_process_group("nccl", device_id=device)
    dtype = torch.float32 if a.dtype == "f32" else torch.float64
    E, N, K, W = a.envs_per_gpu, a.agents, a.steps, max(a.warmup, 3)
    lo, hi = fgd.shard_range(E * world, rank, world)              # contiguous env range of this rank
    env = formation_gym.make_batched_env(a.scenario, hi - lo, N, a.episode_length, device=device,
                                         dtype=dtype, seed=0, auto_reset=True, env_offset=lo,
                                         write_obs=not a.no_obs, u_noise=a.u_noise or None)
    env.reset()

    def barrier():
        if world > 1:
            dist.barrier()

    def one_step():
        if a.two_kernels:
            env.sample_actions()
            return env.step(env.actions)
        return env.step_random(record_actions=True)

    for _ in range(W):
        one_step()
    torch.cuda.synchronize()

    # ---- timed region 1 (-> value): EXACTLY K steps, replayed from a CUDA graph of per-step launches
    # (random-policy kernel + fused step kernel per step; the Philox tick lives on the device so every
    # replayed step draws fresh numbers).  Host cost per step ~0, so the number is the GPU's.
    chunk = max(1, min(K, a.graph_steps))
    while K % chunk:
        chunk -= 1
    graph = env.capture_steps(chunk, fused_random=not a.two_kernels) if a.graph_steps > 0 else None
    if graph is not None:
        graph.replay()
    torch.cuda.synchronize()
    # the settle phase below runs for a fixed time, not a fixed number of steps: the state it leaves is put back, so
    # that the timed steps start from the same state and draw the same actions in every run
    snapshot = env_snapshot(torch, env)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    # Untimed settle phase: ~0.3 s of the same steps so that the clock sampler has samples UNDER LOAD and the SM / memory
    # clocks are at their steady state when the timed region starts (an idle 0.3 s wait here let the GPU drop to its
    # idle clocks, and a 1 ms timed region -- 20 steps -- then ran its first steps while they ramped up again).
    settle_steps, t_settle = 0, time.time()
    while time.time() - t_settle < 0.3:
        if graph is not None:
            graph.replay(); settle_steps += chunk
        else:
            one_step(); settle_steps += 1
        if settle_steps % (8 * chunk) == 0:
            torch.cuda.synchronize()
    env_restore(env, snapshot)
    del snapshot
    launches0 = env.launches
    barrier(); torch.cuda.synchronize()
    ev0.record()
    if graph is not None:
        for _ in range(K // chunk):
            graph.replay()
    else:
        for _ in range(K):
            one_step()
    ev1.record()
    torch.cuda.synchronize(); barrier()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, torch, env)
    launches = (2 if a.two_kernels else 1) * K                    # (fg::k_random_actions +) step kernel per step
    ms = ev0.elapsed_time(ev1)

    # ---- timed region 2 (-> roofline): the fused step kernel ALONE.  G steps are captured into a CUDA graph, each
    # on its own pre-sampled action buffer (fresh actions every step, as in region 1, but no random-policy kernel in
    # between), and the graph is replayed until K steps have run; CUDA events on the launching stream bracket the
    # replays.  kernel_ms = elapsed / steps is the kernel's average launch duration including the (sub-microsecond)
    # kernel-to-kernel hand-over inside the graph.  (Events recorded around every single launch, the first version
    # of this region, added ~5 us of launch latency to each 53 us kernel.)
    G = max(1, min(K, 20))
    acts = []
    for _ in range(G):
        env.sample_actions()
        acts.append(env.actions.clone())
        env.step(env.actions)                                     # also advances the state / tick like region 1
    env.use_device_tick(True)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(side):
        for a_k in acts:                                          # warm-up outside capture (per-buffer fg_buffers)
            env.step(a_k)
    torch.cuda.current_stream(device).wait_stream(side)
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        for a_k in acts:
            env.step(a_k)
    g2.replay(); torch.cuda.synchronize()
    reps2 = max(1, (K + G - 1) // G)
    er0, er1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); torch.cuda.synchronize()
    er0.record()
    for _ in range(reps2):
        g2.replay()
    er1.record()
    torch.cuda.synchronize(); barrier()
    region2_ms = er0.elapsed_time(er1)
    kernel_ms = region2_ms / (reps2 * G)
    del g2, acts
    # keep the sampler alive a little if the regions were short, so it has samples under load
    clocks = None
    if sampler:
        t_extra = time.time()
        while len(sampler.rows) < 3 and time.time() - t_extra < 1.0:
            one_step()
        torch.cuda.synchronize()
        clocks = sampler.stop()
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    total_agents = (hi - lo) * world * N
    value = total_agents * K / (ms * 1e-3)

    bytes_per_env_step = env.bytes_per_env_step()
    # episode statistics: the ONLY collective of the design (NCCL all-reduce of 4 doubles)
    stats = fgd.all_reduce_stats(env.stats.clone())
    ep = {"episodes": float(stats[0]), "return_mean": float(stats[1] / stats[0]) if float(stats[0]) else None}

    # ---------------- e2e: the reference-facing VecEnv API with HOST (numpy) buffers ----------------
    # formation_gym.make_vec_env(...).step(actions_np) -> (obs_np, rews_np, dones_np, infos): what the
    # reference's trainers call on SubprocVecEnv (train/maddpg-v2/utils/env_wrappers.py:63-72).  Per step:
    # H2D of the actions from pinned host memory, the fused step kernel, D2H of obs / rewards / dones /
    # individual rewards into pinned host memory, host sync -- all inside the timed region.
    e2e = None
    if env.obs is not None:
        Ke = a.e2e_steps if a.e2e_steps > 0 else max(10, min(K, 100))
        del graph
        venv = formation_gym.make_vec_env(a.scenario, hi - lo, N, a.episode_length, device=device, dtype=dtype,
                                          seed=0, env_offset=lo, to_numpy=True)
        venv.reset()
        act_h = venv.action_buffer                                # pinned host array [E,N,2]
        act_h[...] = torch.empty(act_h.shape, dtype=dtype).uniform_(-1, 1).numpy()
        out_bytes = 0
        for _ in range(2):
            outs = venv.step(act_h)
        out_bytes = outs[0].nbytes + outs[1].nbytes + outs[2].nbytes + outs[3].individual_reward.nbytes
        # bytes that actually cross PCIe per step: the dynamic prefix of every row (whole rows on the 1 step in
        # episode_length that ends the episodes), rewards, dones, individual rewards
        small = outs[1].nbytes + outs[2].nbytes + outs[3].individual_reward.nbytes
        dynf = venv._dyn_items / float(venv._row_items)
        d2h_bytes = small + outs[0].nbytes * (dynf + (1.0 - dynf) / a.episode_length)
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(Ke):
            venv.step(act_h)                                      # returns host arrays (synchronises)
        dt_e = time.perf_counter() - t0
        barrier()
        te = torch.tensor([dt_e], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": total_agents * Ke / float(te.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(act_h.nbytes) * world,
               "d2h_bytes_per_step": int(d2h_bytes) * world,
               "d2h_bytes_full_tensor_per_step": int(out_bytes) * world,
               "cpu_affinity": ("%d cores (NVML ideal affinity of the GPU)" % len(cpus)) if cpus else None,
               "steps": Ke, "api": "formation_gym.make_vec_env(...).step(numpy actions) -> numpy obs/rews/dones/infos",
               "note": "H2D actions + fused step + D2H obs/reward/done/individual reward per step, pinned host buffers, "
                       "host sync every step.  The persistent pinned obs array is kept byte-identical to the device "
                       "tensor by shipping the dynamic prefix of every row (fg_obs_to_host mode 1, 2-D copy engine "
                       "transfer) and whole rows on episode-end steps.  PCIe / host bound: 72-byte row pieces reach "
                       "~24 GB/s useful on this host, the full tensor 55 GB/s"}
        del venv
        # Informational second figure (NOT the `e2e` key): the same VecEnv API with to_numpy=False -- the
        # observations stay in HBM for a policy network on the same GPU; per step the host uploads the actions
        # from pinned memory and reads rewards + dones back.
        try:
            venv = formation_gym.make_vec_env(a.scenario, hi - lo, N, a.episode_length, device=device, dtype=dtype,
                                              seed=0, env_offset=lo, to_numpy=False)
            venv.reset()
            act_p = torch.empty(hi - lo, N, 2, dtype=dtype).uniform_(-1, 1).pin_memory()
            act_d = torch.empty(hi - lo, N, 2, dtype=dtype, device=device)
            rew_p = torch.empty(hi - lo, N, 1, dtype=dtype).pin_memory()
            done_p = torch.empty(hi - lo, N, dtype=torch.bool).pin_memory()

            def dev_step():
                act_d.copy_(act_p, non_blocking=True)
                o, r, d, _ = venv.step(act_d)
                rew_p.copy_(r, non_blocking=True); done_p.copy_(d, non_blocking=True)
                torch.cuda.current_stream(device).synchronize()
            for _ in range(3):
                dev_step()
            Kd = max(10, 5 * Ke)
            barrier(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(Kd):
                dev_step()
            dt_d = time.perf_counter() - t0
            barrier()
            td = torch.tensor([dt_d], dtype=torch.float64, device=device)
            if world > 1:
                dist.all_reduce(td, op=dist.ReduceOp.MAX)
            e2e["obs_on_device"] = {
                "value": total_agents * Kd / float(td.item()), "unit": UNIT, "steps": Kd,
                "h2d_bytes_per_step": int(act_p.numel() * act_p.element_size()) * world,
                "d2h_bytes_per_step": int(rew_p.numel() * rew_p.element_size() + done_p.numel()) * world,
                "api": "make_vec_env(..., to_numpy=False).step(cuda actions) -> CUDA obs; rewards/dones read to host"}
            del venv
        except Exception as ex:                                   # informational only
            e2e["obs_on_device"] = {"error": repr(ex)[:200]}

    del env
    torch.cuda.empty_cache()
    strong, state_hash = None, None
    if not a.no_strong:
        strong, state_hash = strong_scaling(formation_gym, fgd, torch, dist, device, dtype, rank, world, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = hbm_peak()
    # One kernel per step (the default): the timed region of `value` IS a sequence of launches of the dominant kernel
    # (fused step with the in-kernel random policy), so its average launch duration is elapsed / K of that region.
    # Region 2 (the same kernel READING pre-sampled actions from 20 rotating buffers, as with an external policy) is
    # reported beside it.  With --two-kernels the step holds two kernels and region 2 is the step kernel's time.
    reading_ms = kernel_ms
    if not a.two_kernels and a.graph_steps > 0:
        kernel_ms = ms / K
    if strong:
        for row in strong:
            gbs = row.pop("_gbs_per_gpu")
            row["frac_of_hbm_peak_l2_resident_per_gpu" if row["l2_resident"] else "hbm_frac_per_gpu"] = gbs / peak
    bytes_step = bytes_per_env_step * (hi - lo)
    achieved = bytes_step / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tj = json.load(f)
        key = "%s_N%d_E%d_%s" % (a.scenario, N, hi - lo, a.dtype)
        ent = tj.get(key, {})
        traffic = ent.get("dram_bytes_per_launch")
        if traffic is not None:
            traffic_src = ("NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` "
                           "capture of this kernel and launch size on a B200 of this pool, committed as %s (captured %s)"
                           % (ent.get("source"), ent.get("captured", "round 1")))
    except Exception:
        pass
    warp_ns = (3, 4, 5, 6, 7, 8, 9, 16, 25, 27, 32)                # instantiations of k_hd_warp (fg_abi_impl.cuh)
    on_warp = (a.scenario == "formation_hd_env" and N in warp_ns) or (a.scenario == "basic_formation_env" and N == 3)
    kname = ("fg::k_hd_warp<%s,%d,obs=%s,%s> (fg_step_fused, warp-autonomous persistent kernel)"
             % (a.dtype, N, "yes" if not a.no_obs else "no", "hd" if a.scenario == "formation_hd_env" else "basic")) \
        if on_warp else "fg::k_step<%s> (fg_step_fused, tile kernel)" % a.dtype
    roofline = {"bound": "hbm", "kernel": kname,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_env_step": bytes_per_env_step,
                "share_of_step": kernel_ms / (ms / K),
                "reading_actions": {"kernel_ms": reading_ms, "frac": bytes_step / (reading_ms * 1e-3) / 1e9 / peak,
                                    "what": "the same kernel reading pre-sampled actions (20 rotating action buffers, "
                                            "CUDA graph of step launches only) instead of drawing them"},
                "timing": ("CUDA events around the replays of the CUDA graph of the timed region: one launch of this kernel "
                           "per step (random policy drawn and recorded inside it), so kernel_ms = elapsed / steps"
                           if (not a.two_kernels and a.graph_steps > 0) else
                           "CUDA events around replays of a CUDA graph holding only fused-step launches, each on its own "
                           "pre-sampled action buffer (region 1, which gives `value`, runs random-policy kernel + fused "
                           "step per step)")}

    cpu_baseline = None
    if world == 1 and not a.no_cpu_baseline:
        # the UNMODIFIED reference on the host cores (clean subprocess; one env per process), bounded sample
        from oracle import ref_loop_port as rp
        r = reference_cli(a.scenario, N, 0, a.cpu_seconds, None, a.episode_length)
        pr = rp.time_port(a.scenario, N, a.episode_length, seconds=min(a.cpu_seconds, 2.0))
        port = {"value": pr["agent_steps_per_s"], "cores": pr["procs"], "kind": "port",
                "sample": "oracle/ref_loop_port.py, %d processes x %.1f s" % (pr["procs"], min(a.cpu_seconds, 2.0))}
        if r is not None:
            cpu_baseline = {"value": r["agent_steps_per_s"], "unit": UNIT, "cores": r["procs"], "kind": "reference",
                            "sample": "%d processes x %.1f s of per-env stepping (%d env-steps total) of %s N=%d, "
                                      "episode_length %d, random policy; the UNMODIFIED reference (make_env(...).step; "
                                      "files staged by oracle/make_ref.py from /root/reference, run from %s; numpy %s, "
                                      "scipy %s)" % (r["procs"], a.cpu_seconds, r["env_steps"], a.scenario, N,
                                                     a.episode_length, os.path.relpath(r["reference_root"], ROOT)
                                                     if r["reference_root"].startswith(ROOT) else r["reference_root"],
                                                     r["numpy"], r["scipy"]),
                            "port": port}
        else:
            cpu_baseline = dict(port, unit=UNIT)
            cpu_baseline["sample"] += " (no reference tree available: oracle/_ref missing)"

    also = None
    if world == 1 and not a.no_also:
        also = also_configs(formation_gym, torch, device, dtype, peak, a)

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": a.dtype, "data": "synthetic",
        "config": dict(workload_config(a, hi - lo, "gpu"), u_noise=a.u_noise, clock_settle_steps_untimed=settle_steps),
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "clocks": clocks,
        "gpu_launches": launches, "episode_stats": ep, "strong_scaling": strong, "state_hash": state_hash,
        "also": also,
    }
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def flops_per_env_step(N):
    """Algorithmic flops per env-step, SURVEY.md 8(d): F(N) = 27.5 N^2 + 10 N (dense reference arithmetic,
    shared reward terms once per env, no credit removed for early-outs)."""
    return 27.5 * N * N + 10.0 * N


L2_BYTES = 126e6                                                   # B200 L2 (profiling guide)


def _tensor_hash(torch, t, first_elem, salt):
    """Order-independent 64-bit checksum of a tensor slice that is position-dependent in GLOBAL element indices:
    sum_k bits(t[k]) * w(first_elem + k) mod 2^64 with odd weights w -- shards add up to the whole tensor's value."""
    if t.dtype == torch.float32:
        bits = t.contiguous().view(torch.int32).flatten().to(torch.int64) & 0xFFFFFFFF
    elif t.dtype == torch.float64:
        bits = t.contiguous().view(torch.int64).flatten()
    else:
        bits = t.contiguous().flatten().to(torch.int64)
    idx = torch.arange(bits.numel(), dtype=torch.int64, device=t.device) + int(first_elem)
    w = (idx * -7046029254386353131 + int(salt)) | 1               # 0x9E3779B97F4A7C15 as int64; wraps mod 2^64
    return (bits * w).sum()


def strong_scaling(formation_gym, fgd, torch, dist, device, dtype, rank, world, barrier):
    """(1) BASELINE configs[2] (hd N=27, 65536 envs) and configs[3] (hd N=243, 8192 envs) split evenly over the ranks
    (strong scaling: the TOTAL is fixed), whole step = fused step kernel with the in-kernel random policy from a CUDA
    graph, device timed, max over ranks.  (2) state hash: hd N=27, 65536 envs in total, episode_length 10, seed 0, 25 random-policy
    steps (two auto-resets per env): a 64-bit checksum of pos / vel / reward / ideal_shape / ideal_vel / step /
    observations over ALL envs (per-rank partial sums all-reduced) -- Philox is keyed by the global env id, so the
    value must be identical at 1 / 2 / 4 / 8 ranks."""
    rows = []
    for name, N, E_total, steps in (("configs[2] hd N=27, 65536 envs in total", 27, 65536, 50),
                                    ("configs[3] hd N=243, 8192 envs in total", 243, 8192, 20)):
        lo, hi = fgd.shard_range(E_total, rank, world)
        env = formation_gym.make_batched_env("formation_hd_env", hi - lo, N, 25, device=device, dtype=dtype, seed=0,
                                             auto_reset=True, env_offset=lo)
        env.reset()
        g = env.capture_steps(5, fused_random=True)
        g.replay(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        e0.record()
        for _ in range(steps // 5):
            g.replay()
        e1.record()
        torch.cuda.synchronize(); barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item()) / (steps // 5 * 5)
        rows.append({"config": name, "scaling": "strong", "envs_total": E_total, "envs_per_gpu": hi - lo,
                     "n_gpus": world, "agent_steps_per_s": E_total * N / (ms * 1e-3), "ms_per_step": ms,
                     "_gbs_per_gpu": env.bytes_per_env_step() * (hi - lo) / (ms * 1e-3) / 1e9,
                     "l2_resident": env.bytes_per_env_step() * (hi - lo) < L2_BYTES})
        del g, env
        torch.cuda.empty_cache()
    # ---- configs[4] across ranks: env-count sweep points (TOTAL envs fixed, split evenly over the ranks)
    for N in (3, 9, 27):
        for E_total in (16384, 262144, 1048576):
            lo, hi = fgd.shard_range(E_total, rank, world)
            env = formation_gym.make_batched_env("formation_hd_env", hi - lo, N, 25, device=device, dtype=dtype, seed=0,
                                                 auto_reset=True, env_offset=lo)
            env.reset()
            g = env.capture_steps(5, fused_random=True)
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier(); torch.cuda.synchronize()
            e0.record()
            for _ in range(4):
                g.replay()
            e1.record()
            torch.cuda.synchronize(); barrier()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item()) / 20
            rows.append({"config": "configs[4] sweep hd N=%d, %d envs in total" % (N, E_total), "scaling": "strong",
                         "envs_total": E_total, "envs_per_gpu": hi - lo, "n_gpus": world,
                         "agent_steps_per_s": E_total * N / (ms * 1e-3), "ms_per_step": ms,
                         "_gbs_per_gpu": env.bytes_per_env_step() * (hi - lo) / (ms * 1e-3) / 1e9,
                         "l2_resident": env.bytes_per_env_step() * (hi - lo) < L2_BYTES})
            del g, env
            torch.cuda.empty_cache()
    # ---- cross-rank equality check
    N, E_total, T = 27, 65536, 25
    lo, hi = fgd.shard_range(E_total, rank, world)
    env = formation_gym.make_batched_env("formation_hd_env", hi - lo, N, 10, device=device, dtype=dtype, seed=0,
                                         auto_reset=True, env_offset=lo)
    env.reset()
    for _ in range(T):
        env.step_random()
    parts = []
    for salt, (nm, per_env) in enumerate((("pos", N * 2), ("vel", N * 2), ("reward", N), ("ideal_shape", N * 2),
                                          ("ideal_vel", 2), ("step_count", 1), ("obs", N * 6 * N))):
        parts.append(_tensor_hash(torch, getattr(env, nm), lo * per_env, 1000003 * (salt + 1)))
    h = torch.stack(parts)
    if world > 1:
        dist.all_reduce(h, op=dist.ReduceOp.SUM)                   # int64 sums wrap: addition mod 2^64
    tot = 0
    for k, v in enumerate(h.tolist()):
        tot = (tot * 1099511628211 + (v & 0xFFFFFFFFFFFFFFFF)) & 0xFFFFFFFFFFFFFFFF
    state_hash = {"job": "formation_hd_env N=27, 65536 envs in total over %d rank(s), episode_length 10, seed 0, 25 "
                         "in-kernel random-policy steps, auto-reset" % world,
                  "value": "%016x" % tot,
                  "parts": {nm: "%016x" % (v & 0xFFFFFFFFFFFFFFFF) for nm, v in
                            zip(("pos", "vel", "reward", "ideal_shape", "ideal_vel", "step", "obs"), h.tolist())},
                  "how": "sum over all envs of bits(x[k]) * odd_weight(global element index k) mod 2^64 per tensor "
                         "(per-rank partial sums, NCCL all-reduce SUM on int64); must not depend on the rank count"}
    del env
    torch.cuda.empty_cache()
    return rows, state_hash


def _time_graph(torch, graph, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    graph.replay(); torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def also_configs(formation_gym, torch, device, dtype, peak, a):
    """Other BASELINE.json configs, measured briefly (informational; not the headline line).  A line whose step moves
    less than the 126 MB L2 carries `l2_resident: true` and `frac_of_hbm_peak_l2_resident` instead of `hbm_frac`: its
    working set never leaves L2, so the figure is not an HBM roofline fraction."""
    res = []
    fp32_peak = None
    try:
        from formation_gym import probe
        pk = probe.measure("ffma", device=device)                # scalar FFMA probe, CUDA events
        fp32_peak = pk["tflops"]
        res.append({"config": "FP32 peak probe (fg_fp32_probe, scalar FFMA, 8 CTAs/SM)", "tflops": fp32_peak,
                    "ffma2_tflops": probe.measure("ffma2", device=device)["tflops"]})
    except Exception as ex:
        res.append({"config": "FP32 peak probe", "error": repr(ex)[:200]})

    def frac_keys(row, gbs, nbytes_step, key="hbm_frac"):
        if nbytes_step < L2_BYTES:
            row["l2_resident"] = True
            row[key.replace("hbm_frac", "frac_of_hbm_peak_l2_resident")] = gbs / peak
        else:
            row[key] = gbs / peak

    # ---- configs[0]: basic_formation_env, 3 agents / 3 landmarks, ONE env, random policy, episode_length 25 -- the
    # reference's own CPU-runnable case (test.py -r: `python test.py -s basic_formation_env -r`, test.py:14-28 minus
    # render) through the drop-in facade make_env(...).step (fp64 kernels, E = 1), beside the unmodified reference
    # running the same loop on ONE host core.
    try:
        import numpy as np
        fenv = formation_gym.make_env("basic_formation_env", False, 3, 25)
        fenv.seed(0)
        fenv.reset()

        def loop(n):
            for _ in range(n):
                act_n = [space.sample() for space in fenv.action_space]                   # test.py:20
                _, _, done_n, _ = fenv.step(act_n)                                        # test.py:25
                if np.all(done_n):                                                        # test.py:26-27
                    fenv.reset()
        loop(50)
        t0 = time.perf_counter(); loop(500); dt = time.perf_counter() - t0
        row = {"config": "configs[0] basic_formation_env N=3 L=3, 1 env, random policy, episode_length 25: "
                         "formation_gym.make_env(...).step facade (fp64, E=1; test.py -r loop)",
               "env_steps_per_s": 500 / dt, "agent_steps_per_s": 1500 / dt, "us_per_step": dt / 500 * 1e6,
               "launches_per_step": 1, "bound": "host + launch latency (one H2D, one launch, one D2H, one sync per step)"}
        r = reference_cli("basic_formation_env", 3, 1, 2.0, None, 25)
        if r is not None:
            row["cpu_reference_1core"] = {"env_steps_per_s": r["env_steps_per_s"], "agent_steps_per_s": r["agent_steps_per_s"],
                                          "kind": "reference", "sample": "unmodified reference, 1 process x 2 s"}
        res.append(row)
        del fenv
    except Exception as ex:
        res.append({"config": "configs[0] basic_formation_env facade", "error": repr(ex)[:200]})

    def measure(name, scen, N, E, mode, steps, **envkw):
        env = formation_gym.make_batched_env(scen, E, N, 25, device=device, dtype=dtype, seed=1,
                                             write_obs=(mode != "noobs"), **envkw)
        env.reset()
        nbytes = env.bytes_per_env_step() * E
        per_graph = 25 if mode in ("graph", "rollout") else 5
        if mode in ("launch", "launch2"):                         # plain per-step launches: host-bound at small E
            def host_step():
                if mode == "launch2":
                    env.sample_actions(); env.step(env.actions)
                else:
                    env.step_random(record_actions=True)
            for _ in range(5):
                host_step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                host_step()
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
        elif mode == "rollout":
            env.rollout_random(25); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                env.rollout_random(25)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / (steps * 25)
        elif mode == "bfs":
            g = env.capture_steps(5, policy=lambda env_: env_.bfs_actions(3))
            ms = _time_graph(torch, g, max(2, steps // 5)) / 5
            del g
        elif mode == "bfs_fused":                                 # the controller inside the step kernel: one launch per step
            g = env.capture_steps(5, fused_bfs=3)
            ms = _time_graph(torch, g, max(2, steps // 5)) / 5
            del g
        elif mode == "twokernels":                                # round-1 form: policy kernel + step kernel per step
            g = env.capture_steps(5)
            ms = _time_graph(torch, g, max(2, steps // 5)) / 5
            del g
        elif mode == "noobs":
            env.sample_actions()
            g = env.capture_steps(5, policy=lambda env_: None)
            ms = _time_graph(torch, g, max(2, steps // 5)) / 5
            del g
        else:                                                     # "graph" / "step": fused step kernel, in-kernel random policy
            g = env.capture_steps(per_graph, fused_random=True)
            ms = _time_graph(torch, g, max(2, steps // per_graph)) / per_graph
            del g
        gbs = nbytes / (ms * 1e-3) / 1e9
        row = {"config": name, "agent_steps_per_s": E * N / (ms * 1e-3), "ms_per_env_step": ms,
               "algorithmic_GBps": gbs}
        frac_keys(row, gbs, nbytes)
        if mode in ("step", "bfs", "bfs_fused", "twokernels"):
            # the fused step kernel alone (actions pre-sampled, CUDA graph of 5 launches: no launch gaps, no policy
            # kernel) -- the figure comparable with the headline's roofline.frac
            env.sample_actions()
            g5 = env.capture_steps(5, policy=lambda env_: None)
            kms = _time_graph(torch, g5, max(2, steps // 5)) / 5
            row["step_kernel_ms"] = kms
            frac_keys(row, nbytes / (kms * 1e-3) / 1e9, nbytes, "hbm_frac_step_kernel")
            del g5
        if mode == "noobs":
            tf = flops_per_env_step(N) * E / (ms * 1e-3) / 1e12
            row.pop("hbm_frac", None); row.pop("frac_of_hbm_peak_l2_resident", None)
            row.update({"bound": "fp32", "algorithmic_TFLOPs": tf, "fp32_peak_TFLOPs": fp32_peak,
                        "fp32_frac_algorithmic": (tf / fp32_peak) if fp32_peak else None,
                        "flops_per_env_step": flops_per_env_step(N),
                        "fma_pipe_counter": fma_counter(N, E),
                        "note": "fused step kernel alone (actions pre-sampled, CUDA graph of 5 steps); algorithmic flops "
                                "F(N) = 27.5 N^2 + 10 N over the MEASURED scalar-FFMA peak; the hardware counter "
                                "sm__pipe_fma_cycles_active comes from the committed ncu summary named in fma_pipe_counter"})
        del env
        torch.cuda.empty_cache()
        return row

    cfgs = [
        ("configs[1] hd N=9 E=4096 (per-step launches from the host, one fused kernel per step)", "formation_hd_env", 9,
         4096, "launch", 1000, {}),
        ("configs[1] hd N=9 E=4096 (per-step launches from the host, policy kernel + step kernel)", "formation_hd_env", 9,
         4096, "launch2", 1000, {}),
        ("configs[1] hd N=9 E=4096 (CUDA graph of 25 fused steps)", "formation_hd_env", 9, 4096, "graph", 250, {}),
        ("configs[1] hd N=9 E=4096 (in-kernel 25-step rollouts)", "formation_hd_env", 9, 4096, "rollout", 40, {}),
        ("hd N=9 E=131072, u_noise=0.1 (Philox motor noise, core.py:232-236)", "formation_hd_env", 9, 131072, "step", 50,
         dict(u_noise=0.1)),
        ("hd N=9 E=131072, round-1 form: random-policy kernel + step kernel per step (two launches)",
         "formation_hd_env", 9, 131072, "twokernels", 50, {}),
        ("hd N=3 E=1048576", "formation_hd_env", 3, 1048576, "step", 50, {}),
        ("hd N=9 E=131072, device controller get_action_BFS(ezpolicy) instead of the random policy",
         "formation_hd_env", 9, 131072, "bfs", 50, {}),
        ("hd N=3 E=1048576 (test.py's default tree: 3 agents, one layer), device controller kernel + step kernel per step",
         "formation_hd_env", 3, 1048576, "bfs", 30, {}),
        ("hd N=3 E=1048576, device controller compiled INTO the step kernel (fg_step_policy: one launch per step)",
         "formation_hd_env", 3, 1048576, "bfs_fused", 30, {}),
        ("hd N=4 E=262144 (the reference's most used training size: train/README.md:37,49,167)", "formation_hd_env", 4,
         262144, "step", 50, {}),
        ("configs[2] hd N=27 E=65536", "formation_hd_env", 27, 65536, "step", 50, {}),
        ("configs[3] hd N=243 E=1024 (one GPU's share of 8192)", "formation_hd_env", 243, 1024, "step", 30, {}),
        ("configs[3] hd N=243 E=8192 (all 8192 envs on one GPU)", "formation_hd_env", 243, 8192, "step", 10, {}),
        ("hd N=243 E=1024 state+reward only (no obs)", "formation_hd_env", 243, 1024, "noobs", 20, {}),
        ("hd N=243 E=8192 state+reward only (no obs)", "formation_hd_env", 243, 8192, "noobs", 10, {}),
        ("hd N=81 E=8192", "formation_hd_env", 81, 8192, "step", 20, {}),
        ("basic N=3 L=3 E=1048576", "basic_formation_env", 3, 1048576, "step", 50, {}),
        # SURVEY.md 8(f) rank 3, at the sizes the reference's training recipes use (train/README.md:40-53,167-173: 4 / 5
        # agents, make_world's default landmark counts): fg::k_lm_warp (fg_warp_lm.cuh)
        ("formation_hd_partial_env N=4 L=5 num_obs=3 E=262144 (train/README.md:51)", "formation_hd_partial_env", 4, 262144,
         "step", 50, {}),
        ("formation_hd_partial_env N=5 L=5 num_obs=3 E=262144 (train/README.md:40)", "formation_hd_partial_env", 5, 262144,
         "step", 50, {}),
        ("formation_hd_partial_range_env N=4 L=4 E=262144", "formation_hd_partial_range_env", 4, 262144, "step", 50, {}),
        ("formation_hd_obs_env N=4, 4 goals + 3 obstacles, E=262144 (train/README.md:43,171)", "formation_hd_obs_env", 4,
         262144, "step", 50, {}),
    ]
    for name, scen, N, E, mode, steps, kw in cfgs:
        try:
            res.append(measure(name, scen, N, E, mode, steps, **kw))
        except Exception as ex:  # keep the headline line alive
            res.append({"config": name, "error": repr(ex)[:200]})
    # ---- configs[4]: env-count sweep 1K .. 1M envs x {3, 9, 27} agents on this GPU (whole step = fused step kernel with
    # the in-kernel random policy, from a CUDA graph; the step kernel on pre-sampled actions next to it).  The reference's own scale is 128-200 env processes
    # (train/mappo/train_formation.sh:13); the launch-bound -> HBM-bound crossover shows here.
    sweep = []
    for N in (3, 9, 27):
        for E in (1024, 4096, 16384, 65536, 262144, 1048576):
            try:
                r = measure("sweep", "formation_hd_env", N, E, "step", 25 if E >= 262144 else 50)
                r.pop("config")
                sweep.append(dict({"N": N, "E": E}, **r))
            except Exception as ex:
                sweep.append({"N": N, "E": E, "error": repr(ex)[:200]})
    res.append({"config": "configs[4] env-count sweep, formation_hd_env, 1 GPU (per-N multi-GPU points: the SCALE runs "
                          "are weak scaling, i.e. E per GPU fixed)", "rows": sweep})
    return res


def fma_counter(N, E):
    """sm__pipe_fma_cycles_active (hardware counter) of the no-obs step kernel from the committed ncu summary, if
    one exists for this size: bench.py cannot run ncu itself, so the figure is quoted with its source."""
    try:
        with open(os.path.join(ROOT, "profiles", "fma_pipe.json")) as f:
            return json.load(f).get("hd_N%d_E%d_noobs" % (N, E))
    except Exception:
        return None


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
