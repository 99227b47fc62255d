"""StateReplayBuffer -- an off-policy replay buffer (MADDPG: train/maddpg-v1 .. v5) that stores transitions as env
STATE and decodes the sampled observations on the device.

An observation row is made of copies and single subtractions of the env state (pos, vel, comm, and ideal_shape /
ideal_vel or the landmarks), so ``[N, D]`` observations are a function of about 5N state items.  Storing states instead
of ``obs`` and ``next_obs`` shrinks a transition by 2.4x at formation_hd_env N = 3 and 22x at N = 27 (DESIGN.md 3.3);
``sample`` turns the records back into observation rows with one ``fg_obs_gather`` launch, bit-identical to what the
steps returned.
"""
import ctypes as C
import math

import torch

from . import _native as nat


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
        """Next ring slot; drops its own transition and the one whose s it held.  Returns the slot and the slot of the
        dropped child transition (-1: none)."""
        j = self._next
        self._valid.pop(j, None)
        c = self._child[j]
        dropped = -1
        if c >= 0 and self._prev[c] == j and self._prev_stamp[c] == self._stamp[j]:
            dropped = c if self._valid.pop(c, None) is not None else -1
        self._child[j] = -1
        self._writes += 1
        self._stamp[j] = self._writes
        self._next = (j + 1) % self.capacity
        self._valid_dev = None
        return j, dropped

    def mark_start(self):
        """Snapshot the env's current state into the next slot as the start of a chain (no transition)."""
        j, _ = self._claim()
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
        j, _ = self._claim()
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


class _PrioritizedBatch(dict):
    """A ``PrioritizedStateReplayBuffer.sample`` result: a dict that remembers the buffer it came from."""
    __slots__ = ("buffer",)


class PrioritizedStateReplayBuffer(StateReplayBuffer):
    """``StateReplayBuffer`` with proportional prioritized replay (PER, Schaul et al. 2016; the defaults are baselines'
    ``PrioritizedReplayBuffer``): transition (slot j, env e) is drawn with probability ``p_je / sum p`` and weighted by
    ``w = (min p / p_je) ** beta``, i.e. ``(N P)^-beta / max w``.

    The priorities live on the device in a 32-ary sum/min tree (include/formation_gym_b200.h ``fg_per``): one fp64 leaf
    per transition, 8.5 bytes per transition with the inner nodes, plus 4 bytes of update scratch.  ``add`` gives the
    new transitions the largest priority written so far (initially 1), ``mark_start`` and the transitions a write drops
    get 0.  A sample is one ``fg_per_sample`` launch (tree descent, weights, actions, reward, done and the record rows)
    and one ``fg_obs_gather``; an update is a few launches; neither synchronises.

    Usage::

        buf = PrioritizedStateReplayBuffer(env, capacity, alpha=0.6)
        env.reset(); buf.mark_start()
        for t in range(steps):
            env.step(act); buf.add(act)
            b = buf.sample(B, beta)                    # + weights, index, stamp
            td = q(b['obs'], b['actions']) - target(b)
            loss = (b['weights'] * td ** 2).mean()
            buf.update_priorities(b, td.detach())      # [B] fp32 / fp64: new priority (|td| + eps) ** alpha

    An update entry whose transition was overwritten or dropped since the sample (the slot's stamp changed), or whose
    td is NaN / inf, changes nothing; among entries for one transition the last one wins.

    ``priorities`` is a view of the device leaves, so reading it costs nothing; it is for reading only.  The inner nodes
    are not recomputed from a write through it, so the tree would then no longer sum its leaves: change priorities
    with ``update_priorities`` (or ``.clone()`` the view before editing a copy).
    """

    def __init__(self, env, capacity, alpha=0.6, eps=1e-6):
        alpha, eps = float(alpha), float(eps)
        if not (math.isfinite(alpha) and alpha >= 0):
            raise ValueError("alpha must be finite and >= 0, got %r" % alpha)
        if not (math.isfinite(eps) and eps > 0):
            raise ValueError("eps must be finite and > 0, got %r" % eps)
        super().__init__(env, capacity)
        self.alpha, self.eps = alpha, eps
        T, E = self.capacity, env.E
        self._lib = nat.load()
        nodes, depth, scratch = C.c_longlong(), C.c_int(), C.c_longlong()
        nat.check(self._lib.fg_per_layout(T, E, C.byref(nodes), C.byref(depth), C.byref(scratch)), "fg_per_layout")
        self.depth = depth.value
        kw = dict(device=env.device, dtype=torch.float64)
        self._leaf = torch.zeros(T * E, **kw)
        self._sum = torch.zeros(nodes.value, **kw)
        self._min = torch.full((nodes.value,), float("inf"), **kw)
        self._max_leaf = torch.ones(1, **kw)
        self._stamp_dev = torch.zeros(T, dtype=torch.int64, device=env.device)
        self._prev_dev = torch.full((T,), -1, dtype=torch.int64, device=env.device)
        self._scratch = torch.zeros(scratch.value // 4, dtype=torch.int32, device=env.device)
        t = self._tree = nat.fg_per()
        for k in ("leaf", "sum", "min", "max_leaf", "scratch"):
            setattr(t, k, nat.ptr(getattr(self, "_" + k)))
        t.stamp, t.prev = nat.ptr(self._stamp_dev), nat.ptr(self._prev_dev)
        t.slots, t.envs = T, E
        self._dropped = -1

    @property
    def priorities(self):
        """The leaves as a ``[T, E]`` fp64 view (0 where no transition).  Read-only by contract: a write through it
        bypasses the tree (see the class docstring)."""
        return self._leaf.view(self.capacity, self.env.E)

    def _claim(self):
        j, self._dropped = super()._claim()
        return j, self._dropped

    def _fill(self, valid):
        j, env = self._head, self.env
        with env._on_device():
            rc = self._lib.fg_per_fill(C.byref(self._tree), j, self._prev[j], self._stamp[j], int(valid), self._dropped,
                                       env._stream())
        nat.check(rc, "fg_per_fill")

    def mark_start(self):
        super().mark_start()
        self._fill(False)

    def add(self, actions):
        super().add(actions)
        self._fill(True)

    def sample(self, batch_size, beta=0.4, generator=None):
        """``batch_size`` transitions drawn in proportion to their priorities (with replacement), on the device.
        Returns the keys of ``StateReplayBuffer.sample`` plus ``weights`` [B] (env dtype, ``(min p / p) ** beta``) and
        ``index``, ``stamp`` [B] (int64; what ``update_priorities`` reads).  No host synchronisation."""
        B = int(batch_size)
        if B < 1:
            raise ValueError("batch_size must be >= 1")
        beta = float(beta)
        if not (math.isfinite(beta) and beta >= 0):
            raise ValueError("beta must be finite and >= 0, got %r" % beta)
        if not self._valid:
            raise ValueError("the buffer holds no transition (mark_start(), then step and add())")
        env = self.env
        dev, dt = env.device, env.dtype
        u = torch.rand(B, dtype=torch.float64, generator=generator, device=dev)
        ids = torch.empty(6, B, dtype=torch.int64, device=dev)       # rows (s, s'), index, stamp, slot, env
        done = torch.empty(B, dtype=torch.bool, device=dev)
        w = torch.empty(B, dtype=dt, device=dev)
        act = torch.empty(B, env.N, env.act_dim, dtype=dt, device=dev)
        rew = torch.empty(B, env.N, dtype=dt, device=dev)
        P = nat.ptr
        with env._on_device():
            rc = env._fn("fg_per_sample")(C.byref(self._tree), P(u), B, beta, P(self.done), P(self.actions),
                                          P(self.reward), env.N, env.act_dim, P(ids[0]), P(ids[2]), P(ids[3]),
                                          P(ids[4]), P(ids[5]), P(done), P(w), P(act), P(rew), env._stream())
        nat.check(rc, "fg_per_sample")
        obs = env.gather_observations(self.states, ids[:2].view(-1))
        out = _PrioritizedBatch(obs=obs[:B], next_obs=obs[B:], actions=act, reward=rew, done=done, env_index=ids[5],
                                slot=ids[4], weights=w, index=ids[2], stamp=ids[3])
        out.buffer = self
        return out

    def update_priorities(self, batch, td_errors):
        """Set the priorities of the transitions of ``batch`` (a ``sample`` result of this buffer) to
        ``clamp((|td| + eps) ** alpha, 2**-1022, 2**960)``; ``td_errors`` is an fp32 / fp64 device tensor [B] (a
        per-agent critic reduces its errors to one per transition first).  Entries whose transition was overwritten or
        dropped since the sample, and NaN / inf entries, are skipped.  No host synchronisation."""
        if not isinstance(batch, _PrioritizedBatch) or batch.buffer is not self:
            raise ValueError("batch must be a sample() result of this buffer")
        index, stamp = batch.get("index"), batch.get("stamp")
        if not (torch.is_tensor(index) and torch.is_tensor(stamp) and index.dtype == stamp.dtype == torch.int64
                and index.dim() == 1 and index.shape == stamp.shape and index.is_contiguous() and stamp.is_contiguous()
                and index.device == stamp.device == self.env.device):
            raise ValueError("batch['index'] / batch['stamp'] must be the int64 [B] device tensors sample() returned")
        B = int(index.shape[0])
        if not torch.is_tensor(td_errors) or td_errors.dtype not in (torch.float32, torch.float64):
            raise ValueError("td_errors must be a float32 or float64 tensor")
        if tuple(td_errors.shape) != (B,):
            raise ValueError("td_errors must have shape %s, got %s" % ((B,), tuple(td_errors.shape)))
        if td_errors.device != self.env.device:
            raise ValueError("td_errors must be on %s, got %s" % (self.env.device, td_errors.device))
        td = td_errors.contiguous()
        env = self.env
        with env._on_device():
            rc = self._lib.fg_per_update(C.byref(self._tree), nat.ptr(index), nat.ptr(stamp), nat.ptr(td),
                                         int(td.dtype == torch.float64), B, self.alpha, self.eps, env._stream())
        nat.check(rc, "fg_per_update")
