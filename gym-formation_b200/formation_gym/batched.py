"""BatchedFormationEnv -- thousands to millions of gym-formation envs as contiguous
``[envs, agents, dim]`` device tensors, stepped by ONE fused sm_100a kernel per step.

Shape contract = the reference's VecEnv wrappers (train/maddpg-v2/utils/env_wrappers.py:14-18,
68-72; train/maddpg-v4/runner.py:204): ``obs[E,N,D]  rews[E,N,1]  dones[E,N]`` and auto-reset
when the episode ends (terminal reward/done returned together with the RESET observation).

Semantics of one ``step(actions)`` = ``MultiAgentEnv.step`` of the reference
(formation_gym/environment.py:113-142) for every env: ``_set_action`` (u = a * 5), ``World.step``
(formation_gym/core.py:206-225), scenario ``observation`` / ``reward`` for every agent
(formation_gym/envs/formation_hd_env.py:38-75, basic_formation_env.py:29-52), ``done`` and the
shared-reward sum.  All of it runs in the CUDA library behind include/formation_gym_b200.h;
this class only owns tensors and calls the C ABI.  There is no CPU path.
"""
import ctypes as C

import torch

import contextlib

from . import _native as nat

_NULL_CTX = contextlib.nullcontext()

SCENARIOS = {"formation_hd_env": nat.FG_SCENARIO_HD, "basic_formation_env": nat.FG_SCENARIO_BASIC,
             "formation_hd_partial_env": nat.FG_SCENARIO_HD_PARTIAL,
             "formation_hd_partial_range_env": nat.FG_SCENARIO_HD_PARTIAL_RANGE,
             "formation_hd_obs_env": nat.FG_SCENARIO_HD_OBSTACLE}
# scenario defaults: agent size, episode length (formation_hd_env.py:13,26; basic_formation_env.py:18,
# core.py:113)
_DEFAULTS = {"formation_hd_env": dict(agent_size=0.03, world_length=100),
             "basic_formation_env": dict(agent_size=0.1, world_length=50),
             # formation_hd_partial_env.py:15,29 / formation_hd_partial_range_env.py:15,29
             "formation_hd_partial_env": dict(agent_size=0.04, world_length=25, num_landmarks=5),
             "formation_hd_partial_range_env": dict(agent_size=0.04, world_length=25, num_landmarks=4),
             # formation_hd_obs_env.py:14,29: 4 goal landmarks + 3 obstacles
             "formation_hd_obs_env": dict(agent_size=0.1, world_length=50, num_landmarks=4)}


def obs_dim(scenario, num_agents, num_landmarks=3, num_obs=3):
    """Observation length per agent (hd: 6N, formation_hd_env.py:59; basic: 4+2L+4(N-1); partial:
    2+2L+2*num_obs+2(N-1), formation_hd_partial_env.py:66; partial range: 2+2L+4(N-1); obstacle:
    2+2L+4(N-1) with L = goal landmarks + obstacles, formation_hd_obs_env.py:68)."""
    if scenario == "formation_hd_obs_env":
        return 2 + 2 * num_landmarks + 4 * (num_agents - 1)
    if scenario == "formation_hd_env":
        return 6 * num_agents
    if scenario == "formation_hd_partial_env":
        return 2 + 2 * num_landmarks + 2 * num_obs + 2 * (num_agents - 1)
    if scenario == "formation_hd_partial_range_env":
        return 2 + 2 * num_landmarks + 4 * (num_agents - 1)
    return 4 + 2 * num_landmarks + 4 * (num_agents - 1)


def _target_bank(scenario, E, N, shapes, vels, index):
    """Validate a formation_hd_env target bank (include/formation_gym_b200.h fg_targets) on the host: None, or
    (shapes [K,N,2], vels [K,2] or None, index [E] int32 or None) as CPU tensors.  Every reset -- reset() and the
    in-kernel auto-reset -- gives env e the task k = index[e] when that is in [0, K), else a uniform draw:
    ideal_shape = shapes[k] centred as reset_world centres its landmarks (formation_hd_env.py:93), ideal_vel =
    vels[k] (drawn as without a bank when vels is None)."""
    if shapes is None:
        if vels is not None or index is not None:
            raise ValueError("target_vels / target_index need target_shapes")
        return None
    if scenario != "formation_hd_env":
        raise ValueError("target banks are defined for formation_hd_env only (got %r)" % (scenario,))
    shapes = torch.as_tensor(shapes).detach().cpu().to(torch.float64)
    if shapes.dim() != 3 or shapes.shape[0] < 1 or tuple(shapes.shape[1:]) != (N, 2):
        raise ValueError("target_shapes must have shape (K, %d, 2) with K >= 1, got %s" % (N, tuple(shapes.shape)))
    K = int(shapes.shape[0])
    if vels is not None:
        vels = torch.as_tensor(vels).detach().cpu().to(torch.float64)
        if tuple(vels.shape) != (K, 2):
            raise ValueError("target_vels must have shape (%d, 2), got %s" % (K, tuple(vels.shape)))
    if index is not None:
        index = torch.as_tensor(index).detach().cpu()
        if index.dtype.is_floating_point or index.dtype.is_complex or index.dtype == torch.bool:
            raise ValueError("target_index must hold integers, got %s" % index.dtype)
        if tuple(index.shape) != (E,):
            raise ValueError("target_index must have shape (%d,), got %s" % (E, tuple(index.shape)))
        index = index.to(torch.int64).clamp(-1, 2 ** 31 - 1).to(torch.int32)   # out of range stays out of range
    return shapes, vels, index


class BatchedFormationEnv:
    """E independent envs of N agents on one GPU.

    Parameters mirror ``make_env(scenario, benchmark, num_agents, episode_length)`` plus the batch
    size.  ``env_offset`` is the global index of env 0 (multi-GPU sharding: Philox streams are
    keyed by global env id, so results do not depend on the number of ranks).
    """

    def __init__(self, scenario="formation_hd_env", num_envs=4096, num_agents=9, episode_length=None,
                 num_landmarks=None, device="cuda", dtype=torch.float32, seed=0, auto_reset=True,
                 env_offset=0, write_obs=True, track_landmarks=False, u_noise=None, c_noise=None,
                 silent=True, collide=True, accel=None, max_speed=None, mass=1.0, agent_size=None,
                 agent_mass=None, agent_sizes=None, agent_accel=None, agent_max_speed=None,
                 walls=(), dt=0.1, damping=0.25, contact_force=1e2, contact_margin=1e-3,
                 sensitivity=5.0, num_obs=3, obs_range=0.7, num_obstacles=3, obstacle_size=0.15,
                 obstacle_mass=1.0, obstacle_floor=-2.2, obstacle_fall_vy=-1.0, target_shapes=None,
                 target_vels=None, target_index=None, record_final=False):
        if scenario not in SCENARIOS:
            raise ValueError("unknown scenario %r (supported: %s)" % (scenario, sorted(SCENARIOS)))
        if dtype not in (torch.float32, torch.float64):
            raise ValueError("dtype must be torch.float32 or torch.float64")
        bank = _target_bank(scenario, int(num_envs), int(num_agents), target_shapes, target_vels, target_index)
        if record_final and not auto_reset:
            raise ValueError("record_final records the state an auto-reset overwrites: it needs auto_reset=True")
        self._lib = nat.load()                      # raises when the CUDA extension is missing
        self._fns = {}
        if not torch.cuda.is_available():
            raise nat.NativeError("no CUDA device: formation_gym has no CPU fallback")
        self.scenario = scenario
        self.scn = SCENARIOS[scenario]
        self.E, self.N = int(num_envs), int(num_agents)
        if num_landmarks is None:
            num_landmarks = _DEFAULTS[scenario].get("num_landmarks", 3)
        self.L = self.N if self.scn == nat.FG_SCENARIO_HD else int(num_landmarks)
        # formation_hd_obs_env: `landmarks` holds the goal landmarks, then the obstacles (world.landmarks order,
        # formation_hd_obs_env.py:31-44); L counts both
        self.num_obstacles = int(num_obstacles) if self.scn == nat.FG_SCENARIO_HD_OBSTACLE else 0
        self.num_goals = self.L
        self.L += self.num_obstacles
        self.num_obs, self.obs_range = int(num_obs), float(obs_range)
        if self.scn == nat.FG_SCENARIO_HD and self.N < 3:
            raise ValueError("formation_hd_env needs num_agents >= 3 (formation_hd_env.py:58)")
        if not (1 <= self.N <= nat.FG_MAX_AGENTS):
            raise ValueError("num_agents must be in [1, %d]" % nat.FG_MAX_AGENTS)
        self.D = obs_dim(scenario, self.N, self.L, self.num_obs)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise nat.NativeError("device must be a CUDA device: there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._dev_index = self.device.index
        self.dtype = dtype
        self._sfx = "" if dtype == torch.float32 else "_f64"
        d = _DEFAULTS[scenario]
        self.world_length = int(episode_length if episode_length is not None else d["world_length"])
        self.silent = bool(silent)
        self.act_dim = 2 if self.silent else 4
        self.auto_reset = bool(auto_reset)
        self.seed_value = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.env_offset = int(env_offset)
        self._tick = 0
        self.params = nat.make_params(
            dt=dt, damping=damping, contact_force=contact_force, contact_margin=contact_margin,
            sensitivity=sensitivity, agent_size=d["agent_size"] if agent_size is None else agent_size,
            mass=mass, accel=accel, max_speed=max_speed, u_noise=u_noise, c_noise=c_noise,
            collide=collide, silent=silent, world_length=self.world_length, walls=walls,
            num_obs=self.num_obs, obs_range=self.obs_range, num_obstacles=self.num_obstacles,
            obstacle_size=obstacle_size, obstacle_mass=obstacle_mass, obstacle_floor=obstacle_floor,
            obstacle_fall_vy=obstacle_fall_vy, num_landmarks=self.L)
        kw = dict(device=self.device, dtype=dtype)
        E, N, L = self.E, self.N, self.L
        # optional per-agent arrays (kept alive here; the params struct stores raw pointers)
        self._per_agent = {}
        for name, field, arr in (("agent_mass", "agent_mass", agent_mass),
                                 ("agent_sizes", "agent_size_arr", agent_sizes),
                                 ("agent_accel", "agent_accel", agent_accel),
                                 ("agent_max_speed", "agent_max_speed", agent_max_speed)):
            if arr is not None:
                vals = [(-1.0 if x is None else float(x)) for x in arr]
                if len(vals) != N:
                    raise ValueError("%s must have num_agents entries" % name)
                t = torch.tensor(vals, **kw)
                self._per_agent[name] = t
                setattr(self.params, field, t.data_ptr())
        # state
        self.pos = torch.zeros(E, N, 2, **kw)
        self.vel = torch.zeros(E, N, 2, **kw)
        self.comm = torch.zeros(E, N, 2, **kw)
        self.landmarks = torch.zeros(E, L, 2, **kw) if (self.scn != nat.FG_SCENARIO_HD or track_landmarks) else None
        # landmark.state.p_vel; only the obstacle entries [:, num_goals:] are live
        self.landmark_vel = torch.zeros(E, L, 2, **kw) if self.scn == nat.FG_SCENARIO_HD_OBSTACLE else None
        self.ideal_shape = torch.zeros(E, N, 2, **kw) if self.scn == nat.FG_SCENARIO_HD else None
        self.ideal_vel = torch.zeros(E, 2, **kw) if self.scn == nat.FG_SCENARIO_HD else None
        self.step_count = torch.zeros(E, dtype=torch.int32, device=self.device)
        # outputs
        self.obs = torch.zeros(E, N, self.D, **kw) if write_obs else None
        self.reward = torch.zeros(E, N, 1, **kw)
        self.indiv = torch.zeros(E, N, **kw)
        self._done_u8 = torch.zeros(E, N, dtype=torch.uint8, device=self.device)
        self.done = self._done_u8.view(torch.bool)
        self.actions = torch.zeros(E, N, self.act_dim, **kw)     # scratch for the random policy
        # episode statistics (device side; all-reduced by formation_gym.distributed)
        self.ep_return = torch.zeros(E, **kw)
        self.ep_collisions = torch.zeros(E, dtype=torch.int32, device=self.device)
        self.stats = torch.zeros(4, dtype=torch.float64, device=self.device)
        self.launches = 0                                        # kernels launched by this object
        # device-side tick (CUDA graphs): [0] is added to the host tick, [1] is the kernels' arrival
        # counter.  Stays zero -- and the host counter advances -- until use_device_tick(True).
        # sticky per-env flag of the reference's failure mode (coincident agents -> NaN state, core.py:312 /
        # train/README.md:194-197); set by the kernels, cleared by reset() / clear_nan_flags()
        self.nan_flag = torch.zeros(E, dtype=torch.uint8, device=self.device)
        self._tick_dev = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._device_tick = False
        self._ext_bufs = None
        self._bfs_primed = 0          # fan-out n while self.actions holds the controller's output for the current state (step_bfs)
        self._bufs = self._make_buffers()
        self._set_target_bank(bank)
        self._set_final_block(bool(record_final))

    # ------------------------------------------------------------------ plumbing
    def _make_buffers(self, act=None, obs="default"):
        b = nat.fg_buffers()
        b.pos, b.vel = nat.ptr(self.pos), nat.ptr(self.vel)
        b.act = nat.ptr(act) if act is not None else nat.ptr(self.actions)
        # silent agents: c == 0 always (core.py:281-282) and self.comm stays the zeros it was created with, so the
        # kernels need not store it every step (8N B per env-step, 6 % of the traffic at N = 3)
        b.comm = None if self.silent else nat.ptr(self.comm)
        b.ideal_shape, b.ideal_vel = nat.ptr(self.ideal_shape), nat.ptr(self.ideal_vel)
        b.landmarks = nat.ptr(self.landmarks)
        b.landmark_vel = nat.ptr(self.landmark_vel)
        b.step = nat.ptr(self.step_count)
        b.obs = nat.ptr(self.obs) if obs == "default" else nat.ptr(obs)
        b.reward, b.indiv, b.done = nat.ptr(self.reward), nat.ptr(self.indiv), nat.ptr(self._done_u8)
        b.ep_return, b.ep_collisions = nat.ptr(self.ep_return), nat.ptr(self.ep_collisions)
        b.stats = nat.ptr(self.stats)
        b.tick_dev = nat.ptr(self._tick_dev) if self._device_tick else None
        b.nan_flag = nat.ptr(self.nan_flag)
        return b

    def _set_target_bank(self, bank):
        """Device copies of a validated target bank (``_target_bank``) and the fg_targets block that points at them."""
        self.target_shapes = self.target_vels = self.target_index = None
        self._targets = None
        if bank is None:
            return
        shapes, vels, index = bank
        kw = dict(device=self.device, dtype=self.dtype)
        if index is None:
            index = torch.full((self.E,), -1, dtype=torch.int32)            # every reset draws
        # kept alive here: the struct holds raw pointers.  target_index may be rewritten in place between calls (a
        # curriculum); the next reset reads it in stream order.
        self.target_shapes = shapes.to(**kw).contiguous()
        self.target_vels = None if vels is None else vels.to(**kw).contiguous()
        self.target_index = index.to(device=self.device).contiguous()
        t = nat.fg_targets()
        t.shapes, t.vels = nat.ptr(self.target_shapes), nat.ptr(self.target_vels)
        t.index, t.count = nat.ptr(self.target_index), int(shapes.shape[0])
        self._targets = t

    def _set_final_block(self, on):
        """Terminal block (include/formation_gym_b200.h fg_final): ``final_*`` tensors shaped like the state.  An
        auto-resetting step copies into them the post-step state of every env whose episode it ends (``done[:, 0]``),
        before the reset overwrites it; the entries of other envs keep what they held."""
        self.record_final = on
        self.final_pos = self.final_vel = self.final_comm = None
        self.final_ideal_shape = self.final_ideal_vel = self.final_landmarks = None
        self._final = None
        self._final_obs = None
        if not on:
            return
        kw = dict(device=self.device, dtype=self.dtype)
        E, N, L = self.E, self.N, self.L
        self.final_pos = torch.zeros(E, N, 2, **kw)
        self.final_vel = torch.zeros(E, N, 2, **kw)
        if not self.silent:
            self.final_comm = torch.zeros(E, N, 2, **kw)
        if self.scn == nat.FG_SCENARIO_HD:
            self.final_ideal_shape = torch.zeros(E, N, 2, **kw)
            self.final_ideal_vel = torch.zeros(E, 2, **kw)
        else:
            self.final_landmarks = torch.zeros(E, L, 2, **kw)
        f = nat.fg_final()
        f.pos, f.vel, f.comm = nat.ptr(self.final_pos), nat.ptr(self.final_vel), nat.ptr(self.final_comm)
        f.ideal_shape, f.ideal_vel = nat.ptr(self.final_ideal_shape), nat.ptr(self.final_ideal_vel)
        f.landmarks = nat.ptr(self.final_landmarks)
        self._final = f

    def _call(self, name, *args):
        """Entry point ``name``; with a terminal block ``name + '_final'`` (target bank or NULL, then the block), else
        ``name + '_targets'`` with the target bank appended when one is set.  Resets take no terminal block."""
        if self._final is not None and name != "fg_reset":
            t = C.byref(self._targets) if self._targets is not None else None
            return self._fn(name + "_final")(*args, t, C.byref(self._final))
        if self._targets is not None:
            return self._fn(name + "_targets")(*args, C.byref(self._targets))
        return self._fn(name)(*args)

    def _stream(self):
        # raw cudaStream_t of torch's CURRENT stream on this device (what torch.cuda.current_stream(dev).cuda_stream
        # returns, without building a Stream object: the step path is launch-bound for small batches)
        return C.c_void_p(torch._C._cuda_getCurrentRawStream(self._dev_index))

    def _on_device(self):
        """Context that makes ``self.device`` current; free when it already is (the common case --
        one process per GPU), so a step costs one ctypes call on the host."""
        if torch._C._cuda_getDevice() == self._dev_index:
            return _NULL_CTX
        return torch.cuda.device(self.device)

    def _next_tick(self, n=1, stepping=False):
        """Host part of the Philox tick.  While the device tick is on, the stepping kernels advance
        ``_tick_dev[0]`` themselves and the host part stays frozen (total = host + device)."""
        t = self._tick
        if not (stepping and self._device_tick):
            self._tick = (self._tick + n) & 0xFFFFFFFF
        return t

    def use_device_tick(self, on=True):
        """Keep the step counter that seeds Philox on the DEVICE, so that a CUDA graph holding step
        launches (whose kernel arguments are frozen at capture) draws fresh numbers on every replay.
        Switching it off folds the device count back into the host counter (synchronises)."""
        if not on and self._device_tick:
            self._tick = (self._tick + int(self._tick_dev[0].item())) & 0xFFFFFFFF
            self._tick_dev.zero_()
        self._device_tick = bool(on)
        self._bufs = self._make_buffers()           # the buffer block carries (or drops) the tick pointer
        self._ext_bufs = None

    def _fn(self, name):
        f = self._fns.get(name)
        if f is None:
            f = self._fns[name] = getattr(self._lib, name + self._sfx)
        return f

    def _check_actions(self, actions):
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(actions)
        if actions.device != self.device or actions.dtype != self.dtype:
            actions = actions.to(device=self.device, dtype=self.dtype, non_blocking=True)
        if tuple(actions.shape) != (self.E, self.N, self.act_dim):
            raise ValueError("actions must have shape %s, got %s" %
                             ((self.E, self.N, self.act_dim), tuple(actions.shape)))
        return actions.contiguous()

    # ------------------------------------------------------------------ API
    def seed(self, seed=None):
        """MultiAgentEnv.seed (environment.py:106-110): None -> 1."""
        self.seed_value = (1 if seed is None else int(seed)) & 0xFFFFFFFFFFFFFFFF
        self._tick = 0
        self._tick_dev.zero_()

    def reset(self, mask=None):
        """Scenario.reset_world + current_step = 0 for all (or masked) envs; returns obs [E,N,D]."""
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            if tuple(m.shape) != (self.E,):
                raise ValueError("mask must have shape (E,)")
        self._bfs_primed = 0
        with self._on_device():
            rc = self._call("fg_reset", C.byref(self.params), C.byref(self._bufs), self.scn, self.E, self.N,
                            self.L, nat.ptr(m), self.seed_value, self._next_tick(), self.env_offset, self._stream())
            nat.check(rc, "fg_reset")
            self.launches += 1
        if mask is None:
            self.stats.zero_()
            self.nan_flag.zero_()
        else:
            self.nan_flag.masked_fill_(m.bool(), 0)
        return self.observe()

    def observe(self):
        """Recompute obs / reward / individual rewards from the current state (no stepping)."""
        with self._on_device():
            rc = self._fn("fg_obs_reward")(C.byref(self.params), C.byref(self._bufs), self.scn, self.E,
                                           self.N, self.L, self._stream())
            nat.check(rc, "fg_obs_reward")
            self.launches += 1
        return self.obs

    def world_step(self, actions):
        """``World.step`` only (physics; no observation / reward / done)."""
        actions = self._check_actions(actions)
        b = self._make_buffers(act=actions)
        self._bfs_primed = 0
        with self._on_device():
            rc = self._fn("fg_world_step")(C.byref(self.params), C.byref(b), self.E, self.N,
                                           self.seed_value, self._next_tick(1, True), self.env_offset,
                                           self._stream())
            nat.check(rc, "fg_world_step")
            self.launches += 1

    def step(self, actions):
        """One fused env step.  Returns ``(obs[E,N,D], reward[E,N,1], done[E,N], info)`` with
        ``info['individual_reward'] [E,N]`` (environment.py:130).  Outputs are views of buffers
        owned by this object and are overwritten by the next step."""
        if actions is not self.actions:
            actions = self._check_actions(actions)
        b = self._bufs
        if actions.data_ptr() != self.actions.data_ptr():
            if self._ext_bufs is None or self._ext_bufs[0] != actions.data_ptr():
                self._ext_bufs = (actions.data_ptr(), self._make_buffers(act=actions))
            b = self._ext_bufs[1]
        self._launch_fused(b, 1, 0)
        return self.obs, self.reward, self.done, {"individual_reward": self.indiv}

    def step_random(self, record_actions=False):
        """Random policy (test.py:20) drawn in-kernel from Philox, then the fused step -- ONE launch.
        ``record_actions=True`` also writes the drawn actions into ``self.actions`` (what a trainer's replay
        buffer needs), i.e. the same result as ``sample_actions(); step(self.actions)`` in one kernel."""
        self._launch_fused(self._bufs, 1, 2 if record_actions else 1)
        return self.obs, self.reward, self.done, {"individual_reward": self.indiv}

    def final_observation(self):
        """Terminal observations of the last step: ``obs [E,N,D]`` whose rows of the envs with ``done[:, 0]`` are the
        observation of the state the episode ended in -- bit-identical to what that step returns with
        ``auto_reset=False`` (baselines' ``infos[e]['terminal_observation']``; every episode here ends on the time
        limit, so a value target bootstraps from it).  Rows of other envs are unspecified.  Needs
        ``record_final=True``.  One launch into a buffer owned by this object (allocated on first use, overwritten by
        the next call), no synchronisation: it may be captured in a CUDA graph.  A CTA of envs none of which ended
        exits at once, so a call after a step that ended no episode costs about one launch."""
        if self._final is None:
            raise ValueError("final_observation needs record_final=True")
        if self._final_obs is None:
            self._final_obs = torch.zeros(self.E, self.N, self.D, device=self.device, dtype=self.dtype)
        with self._on_device():
            rc = self._fn("fg_final_obs")(C.byref(self.params), C.byref(self._final), nat.ptr(self._done_u8),
                                          nat.ptr(self._final_obs), self.scn, self.E, self.N, self.L, self._stream())
            nat.check(rc, "fg_final_obs")
            self.launches += 1
        return self._final_obs

    def state_record_keys(self):
        """Names of the state arrays an observation is computed from: ``pos``, ``vel``, ``comm`` (non-silent agents),
        then ``ideal_shape`` and ``ideal_vel`` (formation_hd_env) or ``landmarks`` (every other scenario)."""
        keys = ["pos", "vel"] + ([] if self.silent else ["comm"])
        return keys + (["ideal_shape", "ideal_vel"] if self.scn == nat.FG_SCENARIO_HD else ["landmarks"])

    def gather_observations(self, states, rows, out=None):
        """Observations of sampled state records (``fg_obs_gather``): ``out [B,N,D]`` where slot b holds the rows of
        record ``rows[b]``, bit-identical to what a step returned when that state was current.  ``states`` is a dict
        (or an object with attributes) of record tensors named by ``state_record_keys()``, each shaped like the live
        state with R records in place of E (``ideal_vel [R,2]``, ``landmarks [R,L,2]``); ``rows`` is an int64 device
        tensor [B].  Indices may repeat; one outside [0, R) gives slot b a row block of NaN and reads nothing.  Shapes,
        dtypes and devices are checked before the call; one launch, no synchronisation."""
        get = states.get if isinstance(states, dict) else (lambda k: getattr(states, k, None))
        arrs, R = {}, None
        for k in self.state_record_keys():
            t = get(k)
            if not torch.is_tensor(t):
                raise ValueError("states[%r] must be a tensor" % k)
            if t.dtype != self.dtype:
                raise ValueError("states[%r] must have dtype %s, got %s" % (k, self.dtype, t.dtype))
            if R is None:
                R = int(t.shape[0]) if t.dim() > 0 else 0
            want = {"ideal_vel": (R, 2), "landmarks": (R, self.L, 2)}.get(k, (R, self.N, 2))
            if tuple(t.shape) != want:
                raise ValueError("states[%r] must have shape %s, got %s" % (k, want, tuple(t.shape)))
            if not t.is_contiguous():
                raise ValueError("states[%r] must be contiguous" % k)
            arrs[k] = t
        if R < 1:
            raise ValueError("the state block must hold at least one record")
        if not torch.is_tensor(rows) or rows.dtype != torch.int64 or rows.dim() != 1 or rows.shape[0] < 1:
            raise ValueError("rows must be a non-empty 1-D int64 tensor")
        if not rows.is_contiguous():
            raise ValueError("rows must be contiguous")
        B = int(rows.shape[0])
        if out is not None:
            if not torch.is_tensor(out) or out.dtype != self.dtype or tuple(out.shape) != (B, self.N, self.D):
                raise ValueError("out must be a %s tensor of shape %s" % (self.dtype, (B, self.N, self.D)))
            if not out.is_contiguous():
                raise ValueError("out must be contiguous")
        for name, t in list(arrs.items()) + [("rows", rows)] + ([("out", out)] if out is not None else []):
            if t.device != self.device:
                raise ValueError("%s must be on %s, got %s" % (name, self.device, t.device))
        if out is None:
            out = torch.empty(B, self.N, self.D, device=self.device, dtype=self.dtype)
        f = nat.fg_final()
        for k, t in arrs.items():
            setattr(f, k, nat.ptr(t))
        with self._on_device():
            rc = self._fn("fg_obs_gather")(C.byref(self.params), C.byref(f), R, nat.ptr(rows), B, nat.ptr(out),
                                           self.scn, self.N, self.L, self._stream())
            nat.check(rc, "fg_obs_gather")
            self.launches += 1
        return out

    def nan_envs(self, clear=False):
        """Indices of envs that hit the reference's documented failure mode since the flags were last cleared:
        coincident agents make ``delta_pos / dist`` NaN (core.py:312) and the env's state and rewards stay NaN until
        its next reset (train/README.md:194-197).  Synchronises."""
        idx = torch.nonzero(self.nan_flag, as_tuple=False).flatten()
        if clear:
            self.nan_flag.zero_()
        return idx

    def sample_actions(self, out=None):
        """``[space.sample() for space in env.action_space]`` for every env: U(-1,1), on device.
        Uses the tick of the NEXT step, i.e. exactly what step_random() would draw."""
        if not self.silent:
            raise nat.NativeError("sample_actions supports silent agents only")
        out = self.actions if out is None else out
        with self._on_device():
            rc = self._fn("fg_random_actions")(nat.ptr(out), self.E, self.N, self.seed_value,
                                               self._tick, self.env_offset,
                                               nat.ptr(self._tick_dev) if self._device_tick else None,
                                               self._stream())
            nat.check(rc, "fg_random_actions")
            self.launches += 1
        return out

    def bfs_actions(self, num_agents_per_layer=3, out=None):
        """``get_action_BFS(ezpolicy, obs_n, num_agents_per_layer)`` of the reference
        (formation_gym/__init__.py:19-98; the demo policy of test.py:23) for every env, on the device, from
        the current state.  Writes and returns ``self.actions`` (or ``out``) [E,N,2]."""
        if self.scn != nat.FG_SCENARIO_HD:
            raise nat.NativeError("the hand-written controller is defined for formation_hd_env observations")
        if not self.silent:
            raise nat.NativeError("bfs_actions supports silent agents only (action = [u])")
        out = self.actions if out is None else out
        with self._on_device():
            rc = self._fn("fg_policy_bfs")(nat.ptr(self.pos), nat.ptr(self.ideal_shape), nat.ptr(self.ideal_vel),
                                           nat.ptr(out), self.E, self.N, int(num_agents_per_layer),
                                           self._stream())
            nat.check(rc, "fg_policy_bfs")
            self.launches += 1
        return out

    def step_bfs(self, num_agents_per_layer=3, n_steps=1):
        """The reference's demo loop body (test.py:23-25) -- ``act_n = get_action_BFS(ezpolicy, obs_n, n)`` then
        ``env.step(act_n)`` -- for every env, ``n_steps`` times.  ``self.actions`` carries the controller's output
        from one call to the next: the step runs on it, and the kernel refills it from the NEW state (the reset state
        for envs whose episode just ended), so on return it holds the actions the controller gives for the returned
        observations.  One launch per step where the warp-autonomous kernel has the controller compiled in
        (``fg_step_policy``; N = 3 with 3 agents per layer, 4 / 8 with 2, 16 with 4), the step kernel
        + the controller kernel otherwise -- same results.  The first call after anything else changed the state
        (reset, step, load_state_dict, ...) computes the first actions with ``bfs_actions`` (one extra launch)."""
        if self._final is not None and int(n_steps) != 1:
            raise ValueError("record_final: one step per call (done[:, 0] is the mask of the recorded envs)")
        n = int(num_agents_per_layer)
        if self.scn != nat.FG_SCENARIO_HD or not self.silent:
            raise nat.NativeError("the hand-written controller is defined for formation_hd_env with silent agents")
        if self._bfs_primed != n:
            self.bfs_actions(n)
        n_steps = int(n_steps)
        with self._on_device():
            rc = self._call("fg_step_policy", C.byref(self.params), C.byref(self._bufs), self.scn, self.E, self.N,
                            self.L, n_steps, n, int(self.auto_reset), self.seed_value,
                            self._next_tick(n_steps, True), self.env_offset, self._stream())
            nat.check(rc, "fg_step_policy")
            self.launches += 1                 # (calls; a configuration without a fused instantiation launches 2 per step)
        self._bfs_primed = n
        return self.obs, self.reward, self.done, {"individual_reward": self.indiv}

    def rollout_random(self, n_steps):
        """``n_steps`` random-policy steps in ONE launch with the state held on chip; obs / reward /
        done buffers hold the last step's values afterwards."""
        if self._final is not None and int(n_steps) != 1:
            raise ValueError("record_final: one step per call (done[:, 0] is the mask of the recorded envs)")
        self._launch_fused(self._bufs, int(n_steps), 1)
        return self.obs, self.reward, self.done, {"individual_reward": self.indiv}

    def _launch_fused(self, bufs, n_steps, random_actions):
        self._bfs_primed = 0
        with self._on_device():
            rc = self._call("fg_step_fused", C.byref(self.params), C.byref(bufs), self.scn, self.E, self.N,
                            self.L, n_steps, random_actions, int(self.auto_reset), self.seed_value,
                            self._next_tick(n_steps, True), self.env_offset, self._stream())
            nat.check(rc, "fg_step_fused")
            self.launches += 1

    def capture_steps(self, n_steps=1, policy=None, fused_random=False, fused_bfs=0):
        """Capture ``n_steps`` x (policy, fused env step) into ONE CUDA graph and return it; call
        ``graph.replay()`` to run them.  ``policy=None`` is the random policy (test.py:20) written
        into ``self.actions``; otherwise ``policy(env)`` is called during capture and must enqueue,
        on the current stream, whatever fills ``self.actions`` from ``self.obs``.
        ``fused_random=True``: the random policy is drawn AND recorded into ``self.actions`` inside the
        step kernel (``step_random(record_actions=True)``): one launch per step, same results.
        ``fused_bfs=n``: the reference's demo controller with n agents per layer inside the step kernel
        (``step_bfs(n)``).
        Replays cost no host work per step, which is what small batches (launch-bound per step) need.
        Turns the device tick on."""
        self.use_device_tick(True)
        torch.cuda.synchronize(self.device)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))

        def one():
            if fused_bfs:
                self.step_bfs(fused_bfs)
                return
            if fused_random:
                self._launch_fused(self._bufs, 1, 2)
                return
            if policy is None:
                self.sample_actions()
            else:
                policy(self)
            self._launch_fused(self._bufs, 1, 0)

        with torch.cuda.stream(side):          # warm-up outside capture (lazy module loading, statics)
            one()
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(int(n_steps)):
                one()
        return graph

    def render(self, env_index=0, mode='rgb_array', cam_range=None):
        """Render bridge (SURVEY.md 8f rank 4): copy ONE env's state to the host and draw it like the reference's
        viewer (environment.py:243-393): agents half transparent, landmarks / obstacles solid, camera on the
        agents' centroid.  Returns the 700 x 700 x 3 uint8 frame (``mode='human'`` also shows it via pyglet)."""
        from . import render_bridge as rb
        e = int(env_index)
        P = self.pos[e].double().cpu().numpy()
        size = float(self.params.agent_size)
        circles = [(p[0], p[1], size, (0.35, 0.35, 0.85), 0.5) for p in P]
        if self.scn == nat.FG_SCENARIO_HD:
            # landmarks = ideal shape around the agents' centroid (formation_hd_env.py:40-44)
            lm = self.landmarks[e].double().cpu().numpy() if self.landmarks is not None \
                else self.ideal_shape[e].double().cpu().numpy() + P.mean(0)
            circles += [(l[0], l[1], 0.01, (0.25, 0.25, 0.25), 1.0) for l in lm]
        else:
            lm = self.landmarks[e].double().cpu().numpy()
            G = self.num_goals
            circles += [(l[0], l[1], 0.02, (0.0, 0.6, 0.0) if self.num_obstacles else (0.25, 0.25, 0.25), 1.0)
                        for l in lm[:G]]
            circles += [(l[0], l[1], float(self.params.obstacle_size), (0.25, 0.25, 0.25), 1.0) for l in lm[G:]]
        walls = [(rb.wall_rect(w.orient, w.axis_pos, w.end0, w.end1, w.width), (0.0, 0.0, 0.0), 1.0 if w.hard else 0.5)
                 for w in list(self.params.walls)[:self.params.n_walls]]
        center = P.mean(0) if bool((P == P).all()) else (0.0, 0.0)
        frame = rb.rasterize(circles, walls, center, rb.CAM_RANGE if cam_range is None else cam_range)
        if mode != 'rgb_array':
            self._viewer = rb.show(frame, getattr(self, "_viewer", None))
        return frame

    # ------------------------------------------------------------------ bookkeeping
    @property
    def share_obs(self):
        """``obs.reshape(E, -1)`` (train/maddpg-v4/runner.py:204)."""
        return self.obs.reshape(self.E, -1)

    def episode_stats(self):
        """Device-side episode statistics as python floats (synchronises)."""
        n, s, s2, c = self.stats.tolist()
        mean = s / n if n else float("nan")
        return {"episodes": n, "return_sum": s, "return_sq_sum": s2, "collisions": c,
                "return_mean": mean}

    def bytes_per_env_step(self):
        """Algorithmic HBM bytes per env-step (SURVEY.md 8d): B_full(N) = 24N^2 + 53N + 16 for hd
        fp32 with observations; without obs B_state(N) = 53N + 16.  Scaled by the element size."""
        es = 4 if self.dtype == torch.float32 else 8
        N, L = self.N, self.L
        if self.scn == nat.FG_SCENARIO_HD:
            rd = es * (2 * N * 3 + 2 * N + 2) + 4           # act, pos, vel, ideal_shape, ideal_vel, step
        else:
            rd = es * (2 * N * 3 + 2 * L) + 4               # act, pos, vel, landmarks, step
        wr = es * (2 * N * 2 + N) + N + 4                   # pos, vel, reward, done, step
        if self.obs is not None:
            wr += es * N * self.D
        return rd + wr

    def state_dict(self):
        sd = {k: getattr(self, k).clone() for k in
              ("pos", "vel", "comm", "step_count", "ep_return", "ep_collisions", "stats", "nan_flag")}
        for k in ("landmarks", "landmark_vel", "ideal_shape", "ideal_vel", "target_index"):
            if getattr(self, k) is not None:
                sd[k] = getattr(self, k).clone()
        sd["rng"] = {"seed": self.seed_value, "env_offset": self.env_offset,
                     "tick": (self._tick + int(self._tick_dev[0].item())) & 0xFFFFFFFF}
        return sd

    def load_state_dict(self, sd):
        self._bfs_primed = 0
        for k, v in sd.items():
            if k == "rng":
                self.seed_value, self._tick, self.env_offset = v["seed"], v["tick"], v["env_offset"]
                self._tick_dev.zero_()
            else:
                getattr(self, k).copy_(v)
