"""formation_gym -- B200-native drop-in for jc-bao/gym-formation's MPE step path.

    import formation_gym
    env = formation_gym.make_env('formation_hd_env', benchmark=False, num_agents=9, episode_length=25)
    obs_n = env.reset()
    obs_n, reward_n, done_n, info_n = env.step(act_n)

    venv = formation_gym.make_batched_env('formation_hd_env', num_envs=131072, num_agents=9)
    obs = venv.reset(); obs, rew, done, info = venv.step(actions)      # [E,N,*] CUDA tensors

All arithmetic of the step path runs in hand-written sm_100a kernels behind the C ABI in
``include/formation_gym_b200.h``; there is no CPU fallback (importing works without a GPU, any
call that needs the device raises).
"""
import importlib

__all__ = ["make_env", "make_batched_env", "make_vec_env", "ezpolicy", "get_action_BFS", "MultiAgentEnv",
           "BatchedFormationEnv", "CudaVecEnv", "StateReplayBuffer", "PrioritizedStateReplayBuffer", "StateRolloutBuffer",
           "SCENARIOS"]

SCENARIOS = ("basic_formation_env", "formation_hd_env", "formation_hd_partial_env",
             "formation_hd_partial_range_env", "formation_hd_obs_env")


def _load_scenario(scenario_name):
    if scenario_name.endswith(".py"):
        scenario_name = scenario_name[:-3]
    if scenario_name not in SCENARIOS:
        raise ValueError("scenario %r is not part of the accelerated step path (supported: %s)"
                         % (scenario_name, ", ".join(SCENARIOS)))
    return importlib.import_module("formation_gym.envs." + scenario_name).Scenario()


def make_env(scenario_name='basic_formation_env', benchmark=False, num_agents=3, episode_length=None):
    """Reference signature (formation_gym/__init__.py:6) plus the README's 4th argument
    ``episode_length`` (README.md:61).  Returns a ``MultiAgentEnv``."""
    from .environment import MultiAgentEnv
    scenario = _load_scenario(scenario_name)
    if scenario_name == "formation_hd_env" and episode_length is not None:
        world = scenario.make_world(num_agents, episode_length)
    elif scenario_name in ("formation_hd_partial_env", "formation_hd_partial_range_env", "formation_hd_obs_env") \
            and episode_length is not None:
        world = scenario.make_world(num_agents, world_length=episode_length)
    else:
        world = scenario.make_world(num_agents)
        if episode_length is not None:
            world.world_length = episode_length
    if benchmark:
        return MultiAgentEnv(world, scenario.reset_world, scenario.reward, scenario.observation,
                             scenario.benchmark_data, shared_viewer=True)
    return MultiAgentEnv(world, scenario.reset_world, scenario.reward, scenario.observation,
                         shared_viewer=True)


def make_batched_env(scenario_name='formation_hd_env', num_envs=4096, num_agents=9,
                     episode_length=None, **kwargs):
    """Batched front end: ``num_envs`` envs as ``[envs, agents, dim]`` device tensors."""
    from .batched import BatchedFormationEnv
    return BatchedFormationEnv(scenario_name, num_envs, num_agents, episode_length, **kwargs)


def make_vec_env(scenario_name='formation_hd_env', num_envs=128, num_agents=9, episode_length=None, **kwargs):
    """VecEnv-compatible adapter (``SubprocVecEnv`` / ``DummyVecEnv`` interface of the reference's trainers,
    train/maddpg-v2/utils/env_wrappers.py:40-128) over the batched CUDA env."""
    from .vec_env import CudaVecEnv
    return CudaVecEnv(scenario_name, num_envs, num_agents, episode_length, **kwargs)


def _policy_device(pos, shape, ivel, n):
    """One env through the device controller (fg_policy_bfs_f64): pos/shape [N,2], ivel [2] -> act [N,2]."""
    import ctypes as C
    import numpy as np
    import torch
    from . import _native as nat
    lib = nat.load()
    if not torch.cuda.is_available():
        raise nat.NativeError("no CUDA device: formation_gym has no CPU fallback")
    kw = dict(dtype=torch.float64, device="cuda")
    p = torch.as_tensor(np.ascontiguousarray(pos, dtype=np.float64), **kw).reshape(1, -1, 2)
    s_ = torch.as_tensor(np.ascontiguousarray(shape, dtype=np.float64), **kw).reshape(1, -1, 2)
    v = torch.as_tensor(np.ascontiguousarray(ivel, dtype=np.float64), **kw).reshape(1, 2)
    act = torch.empty_like(p)
    rc = lib.fg_policy_bfs_f64(p.data_ptr(), s_.data_ptr(), v.data_ptr(), act.data_ptr(), 1, p.shape[1], int(n),
                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
    nat.check(rc, "fg_policy_bfs_f64")
    return act[0].cpu().numpy()


def ezpolicy(obs):
    """Reference signature (formation_gym/__init__.py:19-47): the hand-written controller of ONE agent from
    its formation_hd_env observation (length 6n).  Evaluated by the device kernel behind ``fg_policy_bfs``:
    the observation is unpacked into an n-agent state in which this agent is the last one (its
    ``current_shape`` row, :31), whose action is the result."""
    import numpy as np
    obs = np.asarray(obs, dtype=np.float64)
    n = len(obs) / 6
    assert n.is_integer(), n
    n = int(n)
    pos = np.concatenate([obs[2:2 * n], [0.0, 0.0]]).reshape(n, 2)          # others, then me at the origin
    shape = obs[4 * n - 2:6 * n - 2].reshape(n, 2)
    return _policy_device(pos, shape, obs[-2:], n)[n - 1]


def _consistent_observations(obs, N):
    """True when every obs[j] (formation_hd_env layout, length 6N) shows the state that obs[0] implies: the same
    ideal shape and ideal velocity, and other_pos == pos[k] - pos[j] for k != j with agent 0 at the origin."""
    import numpy as np
    try:
        O = np.stack([np.asarray(o, dtype=np.float64) for o in obs])
    except ValueError:
        return False
    if O.shape != (N, 6 * N) or not np.all(np.isfinite(O[:, 2:])):
        return False                                                         # malformed / NaN: read them like the reference
    pos = np.concatenate([[0.0, 0.0], O[0, 2:2 * N]]).reshape(N, 2)
    rel = pos[None, :, :] - pos[:, None, :]                                  # rel[j, k] = pos[k] - pos[j]
    keep = ~np.eye(N, dtype=bool)
    want = rel[keep].reshape(N, 2 * (N - 1))                                 # k != j, ascending
    scale = max(1.0, float(np.abs(pos).max()))
    return bool(np.allclose(O[:, 2:2 * N], want, rtol=0.0, atol=1e-9 * scale)
                and np.array_equal(O[:, 4 * N - 2:], O[:1, 4 * N - 2:].repeat(N, 0)))


def get_action_BFS(policy, obs, num_agents_per_layer):
    """Reference signature (formation_gym/__init__.py:49-98): expand ``policy`` hierarchically over the
    per-agent observation list ``obs`` and return the list of actions.

    With ``policy is formation_gym.ezpolicy`` (the reference's demo, test.py:23) the whole tree runs in ONE
    device launch (``fg_policy_bfs_f64``): agent 0's observation gives every position relative to agent 0,
    the ideal shape and the ideal velocity (formation_hd_env.py:52-59).  PRECONDITION of that shortcut: the N
    observations describe ONE consistent state (what ``env.step`` / ``env.reset`` return).  The reference reads
    each layer leader's and each group member's OWN observation, so observations that a wrapper has made
    inconsistent (noise, clipping, per-agent normalisation, stale entries) are detected here -- every
    ``obs[j]``'s other_pos / ideal_shape / ideal_vel slices are compared with the state derived from
    ``obs[0]`` -- and take the host tree walk below, which reads them exactly like the reference does.
    Any other callable is user code: the tree is walked on the host and only ``policy`` itself is called."""
    import numpy as np
    n = int(num_agents_per_layer)
    N = len(obs)
    num_layer = np.log(N) / np.log(n)
    assert num_layer.is_integer(), 'Observation shape error!'
    if policy is ezpolicy and _consistent_observations(obs, N):
        o0 = np.asarray(obs[0], dtype=np.float64)
        pos = np.concatenate([[0.0, 0.0], o0[2:2 * N]]).reshape(N, 2)         # agent 0 at the origin
        act = _policy_device(pos, o0[4 * N - 2:6 * N - 2].reshape(N, 2), o0[-2:], n)
        return [act[i] for i in range(N)]
    queue, act = [[np.asarray(o, dtype=np.float64) for o in obs]], []
    while queue:
        layer_obs = queue.pop(0)
        M = len(layer_obs)
        nxt = M // n
        for i in range(n):
            lead = layer_obs[i * nxt]
            cur = np.insert(lead[2:2 * M], 2 * i * nxt, [0, 0]).reshape(-1, 2)
            cur = np.array([cur[nxt * k:nxt * (k + 1)].mean(axis=0) for k in range(n)])
            cur = np.delete(cur - cur[i], i, 0).flatten()
            ideal = lead[4 * M - 2:6 * M - 2].reshape(-1, 2)
            tgt = np.array([ideal[nxt * k:nxt * (k + 1)].mean(axis=0) for k in range(n)]).flatten()
            obs_in = np.concatenate((lead[:2], cur, [0] * 2 * (n - 1), tgt, lead[-2:]))
            tar_vel = policy(obs_in) * (np.log(M) / np.log(n))
            if nxt == 1:
                act.append(tar_vel)
                continue
            sub = []
            for j in range(i * nxt, (i + 1) * nxt):
                o = layer_obs[j]
                sub.append(np.concatenate((o[:2], o[2:2 * M][2 * i * nxt:2 * (i + 1) * nxt - 2],
                                           [0] * 2 * (nxt - 1),
                                           o[4 * M - 2:6 * M - 2][2 * i * nxt:2 * (i + 1) * nxt], tar_vel)))
            queue.append(sub)
    return act


def __getattr__(name):
    if name == "CudaVecEnv":
        from .vec_env import CudaVecEnv
        return CudaVecEnv
    if name == "StateReplayBuffer":
        from .replay import StateReplayBuffer
        return StateReplayBuffer
    if name == "PrioritizedStateReplayBuffer":
        from .replay import PrioritizedStateReplayBuffer
        return PrioritizedStateReplayBuffer
    if name == "StateRolloutBuffer":
        from .rollout import StateRolloutBuffer
        return StateRolloutBuffer
    if name == "MultiAgentEnv":
        from .environment import MultiAgentEnv
        return MultiAgentEnv
    if name == "BatchedFormationEnv":
        from .batched import BatchedFormationEnv
        return BatchedFormationEnv
    raise AttributeError(name)
