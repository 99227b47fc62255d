"""StateReplayBuffer -- an off-policy replay buffer (MADDPG: train/maddpg-v1 .. v5) that stores transitions as env
STATE and decodes the sampled observations on the device.

An observation row is made of copies and single subtractions of the env state (pos, vel, comm, and ideal_shape /
ideal_vel or the landmarks), so ``[N, D]`` observations are a function of about 5N state items.  Storing states instead
of ``obs`` and ``next_obs`` shrinks a transition by 2.4x at formation_hd_env N = 3 and 22x at N = 27 (DESIGN.md 3.3);
``sample`` turns the records back into observation rows with one ``fg_obs_gather`` launch, bit-identical to what the
steps returned.
"""
import torch


class StateReplayBuffer:
    """Ring of ``capacity`` slots, each holding one batched step of all E envs of ``env`` (a ``BatchedFormationEnv``
    with ``record_final=True``).

    Storage (env dtype, on the env's device): the post-step states ``S[T,E,...]`` and the terminal states ``F[T,E,...]``
    (copied from the env's ``final_*`` block; meaningful where the step ended the episode) form ONE record block of
    ``R = 2 T E`` records, S first -- record ``j E + e`` is S[j, e], record ``T E + j E + e`` is F[j, e] -- and
    ``actions [T,E,N,A]``, ``reward [T,E,N]`` (``reward[..., 0]`` of the step), ``done [T,E]`` (``done[:, 0]``).

    Usage::

        buf = StateReplayBuffer(env, capacity)
        env.reset(); buf.mark_start()
        for t in range(steps):
            act = policy(env.obs)
            env.step(act); buf.add(act)
            batch = buf.sample(B)          # obs, actions, reward, next_obs, done, env_index, slot

    Transition j is ``(s = S[prev[j]], a, r, s' = F[j] if done else S[j], done)``, where ``prev[j]`` is the slot
    written just before j.  ``mark_start()`` starts a new chain: call it after ``reset()``, ``reset(mask)``,
    ``load_state_dict`` or any other edit of the state, so that no transition spans the edit.  Overwriting a slot drops
    the transition whose ``s`` lived there.  Slot bookkeeping is host-side; copies and sampling are enqueued on the
    current stream without synchronisation (``add`` is not CUDA-graph capturable: slot indices are host values).
    """

    def __init__(self, env, capacity):
        if not getattr(env, "record_final", False):
            raise ValueError("StateReplayBuffer needs an env with record_final=True (the terminal states of "
                             "auto-reset episodes)")
        capacity = int(capacity)
        if capacity < 2:
            raise ValueError("capacity must be >= 2 (a transition needs the slot before it), got %d" % capacity)
        self.env, self.capacity = env, capacity
        T, E = capacity, env.E
        self.num_records = 2 * T * E
        kw = dict(device=env.device, dtype=env.dtype)
        shapes = {"ideal_vel": (2,), "landmarks": (env.L, 2)}
        self.states = {k: torch.zeros(self.num_records, *shapes.get(k, (env.N, 2)), **kw)
                       for k in env.state_record_keys()}
        blocks = {k: v.view(2, T, E, *v.shape[1:]) for k, v in self.states.items()}
        self._S = {k: v[0] for k, v in blocks.items()}
        self._F = {k: v[1] for k, v in blocks.items()}
        self.actions = torch.zeros(T, E, env.N, env.act_dim, **kw)
        self.reward = torch.zeros(T, E, env.N, **kw)
        self.done = torch.zeros(T, E, dtype=torch.bool, device=env.device)
        # host bookkeeping: prev[j] = slot of transition j's s (-1: chain start, no transition); stamp[j] = write count
        # of slot j; prev_stamp[j] = stamp of prev[j] when transition j was recorded; child[j] = slot whose s is slot j
        self._prev = [-1] * T
        self._stamp = [0] * T
        self._prev_stamp = [0] * T
        self._child = [-1] * T
        self._writes = 0
        self._next = 0
        self._head = -1                  # slot holding the env's current state, -1 before the first mark_start
        self._valid = {}                 # slot -> prev slot, for every transition whose s still exists
        self._valid_dev = None           # device mirror [V, 2] (slot, prev slot), rebuilt when the set changed

    def __len__(self):
        return len(self._valid) * self.env.E

    def _copy_state(self, j, dst, final):
        env = self.env
        for k, v in dst.items():
            v[j].copy_(getattr(env, ("final_" + k) if final else k))

    def _claim(self):
        """Next ring slot; drops its own transition and the one whose s it held."""
        j = self._next
        self._valid.pop(j, None)
        c = self._child[j]
        if c >= 0 and self._prev[c] == j and self._prev_stamp[c] == self._stamp[j]:
            self._valid.pop(c, None)
        self._child[j] = -1
        self._writes += 1
        self._stamp[j] = self._writes
        self._next = (j + 1) % self.capacity
        self._valid_dev = None
        return j

    def mark_start(self):
        """Snapshot the env's current state into the next slot as the start of a chain (no transition)."""
        j = self._claim()
        self._copy_state(j, self._S, False)
        self._prev[j] = -1
        self._head = j

    def add(self, actions):
        """Record the step just taken: ``actions`` a_t [E,N,A] (what the step ran on), the env's reward, done, post-step
        state and terminal block.  ``step_random(record_actions=True)`` leaves a_t in ``env.actions``; ``step_bfs``
        overwrites ``env.actions`` with the NEXT actions, so pass a copy taken before that call."""
        if self._head < 0:
            raise ValueError("call mark_start() after reset() before the first add()")
        env = self.env
        if tuple(actions.shape) != (env.E, env.N, env.act_dim):
            raise ValueError("actions must have shape %s, got %s" % ((env.E, env.N, env.act_dim), tuple(actions.shape)))
        h = self._head
        j = self._claim()
        self.actions[j].copy_(actions)
        self.reward[j].copy_(env.reward[..., 0])
        self.done[j].copy_(env.done[:, 0])
        self._copy_state(j, self._S, False)
        self._copy_state(j, self._F, True)
        self._prev[j], self._prev_stamp[j] = h, self._stamp[h]
        self._child[h] = j
        self._valid[j] = h
        self._head = j

    def sample(self, batch_size, generator=None):
        """``batch_size`` transitions drawn uniformly (with replacement) from the valid ones, on the device: a uniform
        valid slot times a uniform env.  ``generator``: a torch generator on the env's device (default: torch's).
        Returns a dict of device tensors ``obs``, ``next_obs`` [B,N,D], ``actions`` [B,N,A], ``reward`` [B,N],
        ``done`` [B], ``env_index`` and ``slot`` [B] (int64).  No host synchronisation."""
        B = int(batch_size)
        if B < 1:
            raise ValueError("batch_size must be >= 1")
        if not self._valid:
            raise ValueError("the buffer holds no transition (mark_start(), then step and add())")
        env, E, T = self.env, self.env.E, self.capacity
        if self._valid_dev is None:
            pairs = torch.tensor(sorted(self._valid.items()), dtype=torch.int64)
            self._valid_dev = pairs.pin_memory().to(env.device, non_blocking=True)
        V = self._valid_dev.shape[0]
        k = torch.randint(0, V * E, (B,), device=env.device, generator=generator)
        e = k % E
        pair = self._valid_dev[k // E]
        slot, prev = pair[:, 0], pair[:, 1]
        done = self.done[slot, e]
        here = slot * E + e
        rows = torch.cat([prev * E + e, torch.where(done, here + T * E, here)])
        obs = env.gather_observations(self.states, rows)
        return {"obs": obs[:B], "next_obs": obs[B:], "actions": self.actions[slot, e], "reward": self.reward[slot, e],
                "done": done, "env_index": e, "slot": slot}
