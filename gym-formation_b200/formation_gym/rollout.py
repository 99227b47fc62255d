"""StateRolloutBuffer -- the rollout storage of an on-policy trainer (MAPPO: the reference's train/mappo, which runs the
``onpolicy`` package) that stores the rollout's observations as env STATE, decodes minibatch observations on the device,
and computes GAE advantages and returns in one CUDA launch (``fg_gae``).

``onpolicy``'s ``SharedReplayBuffer`` keeps ``obs [T+1,E,N,D]`` and ``share_obs [T+1,E,N,N*D]``: at formation_hd_env
N = 27 (fp32) that is 17.5 KB + 472 KB per env-step.  A state record is 656 B there, and the observation rows of a
record are recomputed bit-identically by ``fg_obs_gather`` (README, DESIGN.md 3.3g).
"""
import math

import torch

from . import _native as nat


class StateRolloutBuffer:
    """One rollout of ``num_steps`` (T) steps of all E envs of ``env`` (a ``BatchedFormationEnv`` with
    ``auto_reset=True``), on the env's device.

    Storage: ``states``, one block of ``T E`` state records keyed by ``env.state_record_keys()`` -- record ``t E + e``
    is s_t of env e, the state env e's actor saw at step t (the reset state after an auto-reset); ``actions
    [T,E,N,A]``; ``log_probs``, ``rewards`` (``env.reward[..., 0]``), ``advantages``, ``returns`` [T,E,N];
    ``values [T+1,E,N]``; ``done [T,E]`` (bool, ``env.done[:, 0]``); ``final_values [T,E,N]``, allocated at the first
    ``insert`` that passes it (steps inserted without it hold zeros, which GAE treats as a terminal).  Real arrays are
    in the env dtype; ``insert`` converts with ``copy_``.

    Usage::

        buf = StateRolloutBuffer(env, T)
        obs = env.reset(); buf.start()                       # s_0 = the env's current state
        for t in range(T):
            v = critic(obs.reshape(E, -1)).expand(E, N)      # V(s_t)
            a, logp = actor(obs)
            obs, rew, done, info = env.step(a)
            fv = critic(env.final_observation().reshape(E, -1)).expand(E, N)   # record_final=True
            buf.insert(a, logp, v, final_values=fv)          # final_values=None: time limits are terminals
        buf.compute_returns(critic(obs.reshape(E, -1)).expand(E, N), gamma=0.99, gae_lambda=0.95)
        for mb in buf.minibatches(num_mini_batch):           # obs, share_obs, actions, log_probs, values, ...
            ...
        buf.start()                                          # the next rollout starts from the env's current state

    Every episode of this project ends on its time limit.  With ``final_values`` (the critic's value of
    ``env.final_observation()``, the state the episode ended in), the target at a truncation bootstraps from that
    value; without it the truncation is treated as a terminal (``onpolicy``'s default GAE).

    A state edit in the middle of a rollout -- ``reset(mask)``, ``load_state_dict``, writing the state tensors --
    breaks it: the stored record of the next step would not be the state the step started from.  Call ``start()``
    after such an edit.  The buffer only reads the env.  ``insert``, ``compute_returns`` and ``minibatches`` enqueue
    work on the current stream without synchronising with the host, and allocate nothing after the first rollout but
    the tensors they return.
    """

    def __init__(self, env, num_steps):
        num_steps = int(num_steps)
        if num_steps < 1:
            raise ValueError("num_steps must be >= 1, got %d" % num_steps)
        if not getattr(env, "auto_reset", False):
            raise ValueError("StateRolloutBuffer needs an env with auto_reset=True (a rollout runs through episode "
                             "ends)")
        self.env, self.num_steps = env, num_steps
        T, E, N = num_steps, env.E, env.N
        kw = dict(device=env.device, dtype=env.dtype)
        shapes = {"ideal_vel": (2,), "landmarks": (env.L, 2)}
        self.states = {k: torch.zeros(T * E, *shapes.get(k, (N, 2)), **kw) for k in env.state_record_keys()}
        self._S = {k: v.view(T, E, *v.shape[1:]) for k, v in self.states.items()}
        self.actions = torch.zeros(T, E, N, env.act_dim, **kw)
        self.log_probs = torch.zeros(T, E, N, **kw)
        self.rewards = torch.zeros(T, E, N, **kw)
        self.advantages = torch.zeros(T, E, N, **kw)
        self.returns = torch.zeros(T, E, N, **kw)
        self.values = torch.zeros(T + 1, E, N, **kw)
        self.done = torch.zeros(T, E, dtype=torch.bool, device=env.device)
        self.final_values = None
        self._t = -1                     # inserts since start(); -1 before the first start()
        self._ready = False              # compute_returns ran since the last insert

    @property
    def step(self):
        """Steps inserted since ``start()`` (-1 before the first ``start()``)."""
        return self._t

    def _copy_state(self, t):
        env = self.env
        for k, v in self._S.items():
            v[t].copy_(getattr(env, k))

    def start(self):
        """Begin a rollout: record the env's current state as s_0 and forget the previous rollout's steps."""
        self._copy_state(0)
        self._t = 0
        self._ready = False

    def _check(self, name, x, shape):
        env = self.env
        if not torch.is_tensor(x):
            raise ValueError("%s must be a tensor" % name)
        if not x.is_floating_point():
            raise ValueError("%s must be a floating-point tensor, got %s" % (name, x.dtype))
        if tuple(x.shape) != shape:
            raise ValueError("%s must have shape %s, got %s" % (name, shape, tuple(x.shape)))
        if x.device != env.device:
            raise ValueError("%s must be on %s, got %s" % (name, env.device, x.device))

    def insert(self, actions, log_probs, values, final_values=None):
        """Record step t (the ``insert`` count since ``start()``) just taken by the env: ``actions`` [E,N,A] (what the
        step ran on), ``log_probs`` [E,N], ``values`` [E,N] = V(s_t), and ``final_values`` [E,N] (or None) = V of the
        state each episode that ended at this step ended in (read where ``env.done[:, 0]``).  Takes the env's reward
        and done, and its post-step state as s_{t+1}.  Everything is checked before anything is enqueued."""
        if self._t < 0:
            raise ValueError("call start() after reset() before the first insert()")
        if self._t >= self.num_steps:
            raise ValueError("the rollout already holds num_steps = %d steps: compute_returns(), then start()"
                             % self.num_steps)
        env = self.env
        E, N = env.E, env.N
        self._check("actions", actions, (E, N, env.act_dim))
        self._check("log_probs", log_probs, (E, N))
        self._check("values", values, (E, N))
        if final_values is not None:
            self._check("final_values", final_values, (E, N))
        t = self._t
        self.actions[t].copy_(actions)
        self.log_probs[t].copy_(log_probs)
        self.values[t].copy_(values)
        self.rewards[t].copy_(env.reward[..., 0])
        self.done[t].copy_(env.done[:, 0])
        if final_values is not None:
            if self.final_values is None:
                self.final_values = torch.zeros(self.num_steps, E, N, device=env.device, dtype=env.dtype)
            self.final_values[t].copy_(final_values)
        elif self.final_values is not None:
            self.final_values[t].zero_()
        if t + 1 < self.num_steps:
            self._copy_state(t + 1)
        self._t = t + 1
        self._ready = False

    def compute_returns(self, next_values, gamma=0.99, gae_lambda=0.95):
        """GAE over the rollout: ``next_values`` [E,N] = V(s_T) of the env's current state goes to ``values[T]``, then
        one ``fg_gae`` launch writes ``advantages`` and ``returns`` (= advantages + values[:T]).  Needs exactly
        ``num_steps`` inserts since ``start()``; ``gamma`` and ``gae_lambda`` in [0, 1]."""
        if self._t != self.num_steps:
            raise ValueError("compute_returns needs num_steps = %d inserts since start(), got %d"
                             % (self.num_steps, max(self._t, 0)))
        gamma, lam = float(gamma), float(gae_lambda)
        if not (math.isfinite(gamma) and 0.0 <= gamma <= 1.0):
            raise ValueError("gamma must be finite and in [0, 1], got %r" % gamma)
        if not (math.isfinite(lam) and 0.0 <= lam <= 1.0):
            raise ValueError("gae_lambda must be finite and in [0, 1], got %r" % lam)
        env = self.env
        self._check("next_values", next_values, (env.E, env.N))
        self.values[self.num_steps].copy_(next_values)
        P = nat.ptr
        with env._on_device():
            rc = env._fn("fg_gae")(P(self.rewards), P(self.values), P(self.final_values), P(self.done),
                                   P(self.advantages), P(self.returns), self.num_steps, env.E, env.N, gamma, lam,
                                   env._stream())
        nat.check(rc, "fg_gae")
        self._ready = True

    def minibatches(self, num_mini_batch, generator=None):
        """Yield ``num_mini_batch`` minibatches of ``B = (T E) // num_mini_batch`` env-steps drawn without replacement
        from one ``torch.randperm(T E)`` on the device (``generator``: a torch generator on the env's device); the
        remainder is dropped, as ``onpolicy``'s ``feed_forward_generator`` does.  An env-step keeps its N agents
        together.  Each batch is a dict of device tensors: ``obs`` [B,N,D] (decoded from the state records by one
        ``fg_obs_gather``, bit-identical to what the env returned at that step), ``share_obs`` [B,N*D] (a view of
        ``obs``), ``actions`` [B,N,A], ``log_probs``, ``values``, ``returns``, ``advantages`` [B,N], ``step_index`` and
        ``env_index`` [B] (int64).  Needs ``compute_returns`` after the last insert."""
        if not self._ready:
            raise ValueError("call compute_returns() after the rollout's last insert() before minibatches()")
        T, E = self.num_steps, self.env.E
        n = int(num_mini_batch)
        if not 1 <= n <= T * E:
            raise ValueError("num_mini_batch must be in [1, T*E = %d], got %d" % (T * E, n))
        return self._batches(n, generator)

    def _batches(self, n, generator):
        env = self.env
        T, E, N = self.num_steps, env.E, env.N
        B = (T * E) // n
        perm = torch.randperm(T * E, device=env.device, generator=generator)
        flat = {"actions": self.actions.view(T * E, N, env.act_dim), "log_probs": self.log_probs.view(T * E, N),
                "values": self.values[:T].view(T * E, N), "returns": self.returns.view(T * E, N),
                "advantages": self.advantages.view(T * E, N)}
        for i in range(n):
            rows = perm[i * B:(i + 1) * B]                   # a permutation value is the record row t E + e
            obs = env.gather_observations(self.states, rows)
            step = rows.div(E, rounding_mode="floor")
            mb = {"obs": obs, "share_obs": obs.view(B, N * env.D)}
            mb.update({k: v[rows] for k, v in flat.items()})
            mb["step_index"], mb["env_index"] = step, rows - step * E
            yield mb
