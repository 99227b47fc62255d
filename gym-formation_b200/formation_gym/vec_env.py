"""VecEnv-compatible adapter over ``BatchedFormationEnv`` (SURVEY.md section 8f, rank 1).

The reference's trainers never talk to one env: they wrap ``make_env`` in baselines-style vectorised
envs -- one OS process per env, one pickled message per env per step over ``multiprocessing.Pipe``
(train/maddpg-v2/utils/env_wrappers.py:40-128 ``SubprocVecEnv`` / ``DummyVecEnv``;
train/maddpg-v4/wrapper.py:20-131,166-223,407-432 ``ShareVecEnv`` family).  ``CudaVecEnv`` exposes the
same interface -- ``num_envs, observation_space, share_observation_space, action_space, num_agents,
agent_types, reset(), step_async(actions), step_wait(), step(actions), close()`` and the worker's
auto-reset rule (when all agents of an env are done the env is reset and the RESET observation is
returned with the terminal reward / done; env_wrappers.py:14-18, wrapper.py:139-146) -- over ONE fused
kernel launch per step for all envs.

Return types follow the wrappers: ``obs [E,N,D]``, ``rews [E,N,1]``, ``dones [E,N]`` and ``infos``, a
sequence of E per-env lists of N dicts ``{'individual_reward': r}`` (environment.py:130), materialised
lazily.  ``to_numpy=True`` gives what the reference's trainers see -- numpy arrays on the host (pinned
staging buffers, one H2D for the actions and one D2H per output per step); ``to_numpy=False`` keeps
CUDA tensors for device-resident policies (no host round-trip).  There is no CPU path.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as nat
from . import spaces
from .batched import BatchedFormationEnv


class _EnvInfo(object):
    """infos[e]: list-like of N dicts {'individual_reward': r_i} of one env, built on demand; with
    'terminal_observation': agent i's row when the env's episode ended in this step (record_final)."""
    __slots__ = ("_row", "_term")

    def __init__(self, row, term=None):
        self._row = row
        self._term = term

    def __len__(self):
        return len(self._row)

    def __getitem__(self, i):
        if self._term is None:
            return {'individual_reward': float(self._row[i])}
        return {'individual_reward': float(self._row[i]), 'terminal_observation': self._term[i]}

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class InfoBatch(object):
    """``infos`` of one vectorised step.  ``infos[e][i]['individual_reward']`` like the tuple of info
    lists the reference's ``step_wait`` returns (env_wrappers.py:71-72), without creating E*N dicts;
    ``infos.individual_reward`` is the whole ``[E,N]`` array / tensor.  With ``record_final``, on the steps where
    episodes end, ``infos.terminal_observation`` is the whole ``[E,N,D]`` array / tensor of terminal observations
    (rows valid where ``dones[:, 0]``) and ``infos[e][i]['terminal_observation']`` agent i's row, for the envs that
    ended only (the key of baselines' / SB3's VecEnvs, per agent)."""
    terminal_observation = None

    def __init__(self, individual_reward, terminal_observation=None, done=None):
        self.individual_reward = individual_reward
        if terminal_observation is not None:
            self.terminal_observation = terminal_observation
            self._done = done

    def __len__(self):
        return int(self.individual_reward.shape[0])

    def __getitem__(self, e):
        if self.terminal_observation is not None and bool(self._done[e, 0]):
            return _EnvInfo(self.individual_reward[e], self.terminal_observation[e])
        return _EnvInfo(self.individual_reward[e])

    def __iter__(self):
        return (self[e] for e in range(len(self)))


class CudaVecEnv(object):
    """``SubprocVecEnv([make_env(...)] * num_envs)`` of the reference, on one GPU."""
    closed = False
    viewer = None
    metadata = {'render.modes': ['human', 'rgb_array']}

    def __init__(self, scenario_name='formation_hd_env', num_envs=128, num_agents=9, episode_length=None,
                 device="cuda", to_numpy=True, seed=0, **kwargs):
        kwargs.setdefault("auto_reset", True)
        self.env = BatchedFormationEnv(scenario_name, num_envs, num_agents, episode_length, device=device,
                                       seed=seed, **kwargs)
        e = self.env
        if e.obs is None:
            raise ValueError("CudaVecEnv needs observations (write_obs=True)")
        self.num_envs = e.E
        self.num_agents = e.N
        self.to_numpy = bool(to_numpy)
        # per-agent spaces exactly as MultiAgentEnv builds them (environment.py:59-96)
        act_dim = e.act_dim
        self.action_space = [spaces.Box(low=-1.0, high=+1.0, shape=(act_dim,), dtype=np.float32)
                             for _ in range(e.N)]
        self.observation_space = [spaces.Box(low=-np.inf, high=+np.inf, shape=(e.D,), dtype=np.float32)
                                  for _ in range(e.N)]
        self.share_observation_space = [spaces.Box(low=-np.inf, high=+np.inf, shape=(e.N * e.D,),
                                                   dtype=np.float32) for _ in range(e.N)]
        self.agent_types = ['agent' for _ in range(e.N)]          # env_wrappers.py:30-35 (no adversaries)
        self.waiting = False
        self._pending = None
        self._age = None
        self._np_dtype = np.float32 if e.dtype == torch.float32 else np.float64
        # record_final: terminal observations in the infos of the steps where episodes end.  All envs are reset
        # together and share one episode length, so the host knows those steps (None: unknown -> every step)
        self.record_final = e.record_final
        self._final_age = None
        self._final_pending = None
        if self.to_numpy:
            # pinned host staging: actions in, obs / rewards / dones / individual rewards out
            self._act_h = torch.empty(e.E, e.N, act_dim, dtype=e.dtype).pin_memory()
            self._act_d = torch.empty_like(e.actions)
            self._obs_h = torch.empty(e.obs.shape, dtype=e.dtype).pin_memory()
            self._rew_h = torch.empty(e.reward.shape, dtype=e.dtype).pin_memory()
            self._done_h = torch.empty(e.done.shape, dtype=torch.bool).pin_memory()
            self._ind_h = torch.empty(e.indiv.shape, dtype=e.dtype).pin_memory()
            # Only a prefix of every observation row changes from step to step: for silent agents the trailing comm
            # block is zero, and formation_hd_env's [comm | ideal_shape | ideal_vel] (2N of 3N items,
            # formation_hd_env.py:52-59) changes only when the env is reset.  The pinned host array persists, so a
            # step ships that prefix only (fg_obs_to_host mode 1: a 2-D copy-engine transfer) and whole rows on the
            # steps on which the episodes end; the host array stays byte-identical to the device tensor.
            items = e.D // 2
            if e.silent and e.scenario == "formation_hd_env":
                self._dyn_items = e.N
            elif e.silent:
                self._dyn_items = items - (e.N - 1)
            else:
                self._dyn_items = items
            self._row_items = items
            self._age = None                    # env steps since ALL envs were last reset together (None: unknown)
            # What step_wait() / reset() hand out: READ-ONLY numpy views of the persistent pinned buffers.  The obs
            # buffer is refreshed incrementally, so an in-place edit by the caller (e.g. `obs /= scale`) would survive
            # in the part of a row that is not re-sent -- numpy refuses the write instead; copy to modify.
            self._views = tuple(t.numpy() for t in (self._obs_h, self._rew_h, self._done_h, self._ind_h))
            for v in self._views:
                v.flags.writeable = False
            if self.record_final:
                self._fobs_h = torch.empty(e.obs.shape, dtype=e.dtype).pin_memory()
                self._fobs_view = self._fobs_h.numpy()
                self._fobs_view.flags.writeable = False

    # ------------------------------------------------------------------ VecEnv interface
    @property
    def action_buffer(self):
        """(to_numpy) the pinned host array ``step_async`` uploads from; filling it in place and passing
        it to ``step_async`` skips one host copy."""
        return self._act_h.numpy()

    def reset(self):
        """All envs: ``np.stack([env.reset() ...])`` of the wrappers -> obs [E,N,D]."""
        self.waiting = False
        obs = self.env.reset()
        self._age = 0
        self._final_age = 0
        return self._obs_out(obs)

    def reset_task(self):
        raise NotImplementedError("the gym-formation envs define no reset_task()")

    def step_async(self, actions):
        """Enqueue the step of every env (asynchronous on the GPU); ``actions`` is ``[E,N,act_dim]``
        (array-like / tensor), one row per env as ``zip(self.remotes, actions)`` expects
        (env_wrappers.py:63-66)."""
        if self.waiting:
            raise RuntimeError("step_async called while a step is pending")
        e = self.env
        if self.to_numpy and not torch.is_tensor(actions):
            a = np.asarray(actions)
            if a.shape != tuple(self._act_h.shape):
                raise ValueError("actions must have shape %s, got %s" % (tuple(self._act_h.shape), a.shape))
            if a.ctypes.data != self._act_h.data_ptr():
                self._act_h.numpy()[...] = a
            self._act_d.copy_(self._act_h, non_blocking=True)
            actions = self._act_d
        self._pending = e.step(actions)
        self._final_pending = None
        if self.record_final:
            ending = self._final_age is None
            if not ending:
                self._final_age += 1
                ending = self._final_age % e.world_length == 0
            if ending:                                              # episodes (may) end in this step
                self._final_pending = e.final_observation()
                if self.to_numpy:
                    self._fobs_h.copy_(self._final_pending, non_blocking=True)
        if self.to_numpy:                                           # D2H overlaps nothing else: queue it now
            obs, rew, done, info = self._pending
            self._fetch_obs(obs)
            self._rew_h.copy_(rew, non_blocking=True)
            self._done_h.copy_(done, non_blocking=True)
            self._ind_h.copy_(info["individual_reward"], non_blocking=True)
        self.waiting = True

    def step_wait(self):
        """-> (obs [E,N,D], rews [E,N,1], dones [E,N], infos); with ``to_numpy`` the arrays are READ-ONLY views of
        pinned buffers that the next step refreshes (copy them to keep or to modify them)."""
        if not self.waiting:
            raise RuntimeError("step_wait called without step_async")
        self.waiting = False
        obs, rew, done, info = self._pending
        fobs, self._pending, self._final_pending = self._final_pending, None, None
        if self.to_numpy:
            torch.cuda.current_stream(self.env.device).synchronize()
            if fobs is not None:
                return (self._views[0], self._views[1], self._views[2],
                        InfoBatch(self._views[3], self._fobs_view, self._views[2]))
            return (self._views[0], self._views[1], self._views[2], InfoBatch(self._views[3]))
        if fobs is not None:
            return obs, rew, done, InfoBatch(info["individual_reward"], fobs, done)
        return obs, rew, done, InfoBatch(info["individual_reward"])

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def _fetch_obs(self, obs):
        """Queue the D2H transfer of this step's observations into the persistent pinned array.  All envs of a
        CudaVecEnv are reset together and share one episode length, so the steps on which rows change beyond their
        dynamic prefix are known on the host: the steps that end the episodes (auto-reset -> new ideal shape /
        ideal velocity).  Those steps, and any state the host cannot vouch for, take the whole-tensor copy."""
        e = self.env
        whole = self._dyn_items >= self._row_items or self._age is None
        if not whole:
            self._age += 1
            whole = e.auto_reset and (self._age % e.world_length == 0)
        isz = 8 if e.dtype == torch.float32 else 16
        rc = e._lib.fg_obs_to_host(obs.data_ptr(), self._obs_h.data_ptr(), None, None, e.E, e.N, self._row_items,
                                   self._dyn_items, isz, 0 if whole else 1,
                                   C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream))
        nat.check(rc, "fg_obs_to_host")

    def close(self):
        if self.closed:
            return
        if self.waiting:
            self.step_wait()
        self.closed = True

    def render(self, mode='human'):
        """First env of the batch through the render bridge (``BatchedFormationEnv.render``)."""
        return self.env.render(0, mode)

    def seed(self, seed=None):
        self.env.seed(seed)

    @property
    def unwrapped(self):
        return self

    # ------------------------------------------------------------------ helpers for the trainers
    def share_obs(self, obs):
        """``share_obs = obs.reshape(n_rollout_threads, -1)`` -> [E, N*D] (train/maddpg-v4/runner.py:204)."""
        return obs.reshape(self.num_envs, -1)

    def sample_actions(self):
        """``[[space.sample() for space in action_space] for _ in envs]`` (test.py:20), drawn on the device."""
        act = self.env.sample_actions()
        if self.to_numpy:
            self._act_h.copy_(act)
            return self._act_h.numpy()
        return act

    def _obs_out(self, obs):
        if self.to_numpy:
            self._obs_h.copy_(obs)
            return self._views[0]
        return obs


def make_vec_env(scenario_name='formation_hd_env', num_envs=128, num_agents=9, episode_length=None, **kwargs):
    """Factory mirroring ``make_parallel_env`` of the trainers (train/maddpg-v2/main.py:19-30): the
    ``n_rollout_threads`` env processes become one batched CUDA env."""
    return CudaVecEnv(scenario_name, num_envs, num_agents, episode_length, **kwargs)
