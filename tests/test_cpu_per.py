"""Prioritized replay (include/formation_gym_b200.h fg_per_*, formation_gym.replay.PrioritizedStateReplayBuffer), CPU
only: fg_per_layout sizes, every argument rejection of the tree entry points before any device call, and the Python
errors raised before the buffer touches a device."""
import ctypes as C
import math

import pytest
import torch

BASE = 1 << 20                                           # never dereferenced: validation happens first
A64 = BASE + (9 << 12)                                   # an 8-byte aligned address for int64 / fp64 arguments


def _lib():
    from formation_gym import _native as nat
    return nat, nat.load()


def _tree(nat, **kw):
    t = nat.fg_per()
    for k, i in zip(("leaf", "sum", "min", "max_leaf", "stamp", "prev", "scratch"), range(1, 8)):
        setattr(t, k, BASE + (i << 12))
    t.slots, t.envs = 5, 7
    for k, v in kw.items():
        setattr(t, k, v)
    return t


def _host_layout(M):
    nodes, depth, n = 0, 0, M
    while True:
        n = -(-n // 32)
        nodes, depth = nodes + n, depth + 1
        if n == 1:
            return nodes, depth


@pytest.mark.parametrize("slots,envs", [(1, 1), (1, 32), (3, 11), (32, 32), (1, 1025), (5, 7), (100, 65536),
                                        (8, 9 * 131072), (1 << 20, 1 << 20)])
def test_layout_sizes(slots, envs):
    nat, lib = _lib()
    nodes, depth, scratch = C.c_longlong(), C.c_int(), C.c_longlong()
    assert lib.fg_per_layout(slots, envs, C.byref(nodes), C.byref(depth), C.byref(scratch)) == 0
    M = slots * envs
    assert (nodes.value, depth.value) == _host_layout(M)
    assert scratch.value == 4 * M
    if M <= 32:
        assert (nodes.value, depth.value) == (1, 1)
    if M == 100 * 65536:
        assert depth.value == 5                          # 6.5 M leaves


def test_layout_rejections():
    nat, lib = _lib()
    n, d, s = C.c_longlong(), C.c_int(), C.c_longlong()
    cases = [((0, 4, C.byref(n), C.byref(d), C.byref(s)), b"slots and envs must be >= 1"),
             ((4, 0, C.byref(n), C.byref(d), C.byref(s)), b"slots and envs must be >= 1"),
             ((-1, 4, C.byref(n), C.byref(d), C.byref(s)), b"slots and envs must be >= 1"),
             (((1 << 20) + 1, 1 << 20, C.byref(n), C.byref(d), C.byref(s)), b"<= 2^40"),
             ((1 << 62, 4, C.byref(n), C.byref(d), C.byref(s)), b"<= 2^40"),
             ((4, 4, None, C.byref(d), C.byref(s)), b"must be non-null"),
             ((4, 4, C.byref(n), None, C.byref(s)), b"must be non-null"),
             ((4, 4, C.byref(n), C.byref(d), None), b"must be non-null")]
    for args, msg in cases:
        assert lib.fg_per_layout(*args) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and b"fg_per_layout" in err, (msg, err)


def _tree_cases(nat):
    """Malformed trees, rejected by every entry point."""
    cases = [(None, b"the tree must be non-null")]
    for k in ("leaf", "sum", "min", "max_leaf", "stamp", "prev", "scratch"):
        cases.append((_tree(nat, **{k: None}), b"fg_per arrays must be non-null"))
        cases.append((_tree(nat, **{k: BASE + (1 << 12) * 9 + (2 if k == "scratch" else 4)}), b"aligned"))
    cases += [(_tree(nat, slots=0), b"slots and envs must be >= 1"), (_tree(nat, envs=-2), b"slots and envs must be >= 1"),
              (_tree(nat, slots=1 << 21, envs=1 << 20), b"<= 2^40")]
    return cases


def _fill(lib, t, slot=2, prev=1, stamp=3, valid=1, drop=-1):
    return lib.fg_per_fill(C.byref(t) if t is not None else None, slot, prev, stamp, valid, drop, None)


def test_fill_rejections():
    nat, lib = _lib()
    for t, msg in _tree_cases(nat):
        assert _fill(lib, t) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and b"fg_per_fill" in err, (msg, err)
    t = _tree(nat)
    cases = [(dict(slot=-1), b"slot out of range"), (dict(slot=5), b"slot out of range"),
             (dict(prev=-2), b"prev must be -1 or another slot"), (dict(prev=5), b"prev must be -1 or another slot"),
             (dict(prev=2), b"prev must be -1 or another slot"),
             (dict(drop=-2), b"drop_slot must be -1 or another slot"), (dict(drop=5), b"drop_slot must be -1"),
             (dict(drop=2), b"drop_slot must be -1 or another slot"),
             (dict(valid=2), b"valid must be 0 or 1"), (dict(valid=-1), b"valid must be 0 or 1"),
             (dict(prev=-1, valid=1), b"a valid transition needs prev >= 0"), (dict(stamp=-1), b"stamp must be >= 0")]
    for kw, msg in cases:
        assert _fill(lib, t, **kw) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and b"fg_per_fill" in err, (msg, err)


def _update(lib, t, index=A64, stamp=A64 + 4096, td=A64 + 8192, td_f64=0, B=16, alpha=0.6, eps=1e-6):
    return lib.fg_per_update(C.byref(t) if t is not None else None, index, stamp, td, td_f64, B, alpha, eps, None)


@pytest.mark.parametrize("td_f64", [0, 1], ids=["td_f32", "td_f64"])
def test_update_rejections(td_f64):
    nat, lib = _lib()
    for t, msg in _tree_cases(nat):
        assert _update(lib, t, td_f64=td_f64) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and b"fg_per_update" in err, (msg, err)
    t = _tree(nat)
    inf, nan = math.inf, math.nan
    cases = [(dict(B=0), b"B must be >= 1"), (dict(B=-5), b"B must be >= 1"),
             (dict(index=None), b"must be non-null"), (dict(stamp=None), b"must be non-null"),
             (dict(td=None), b"must be non-null"), (dict(td_f64=2), b"td_f64 must be 0 or 1"),
             (dict(index=A64 + 4), b"aligned"), (dict(stamp=A64 + 4), b"aligned"), (dict(td=A64 + 2), b"aligned"),
             (dict(alpha=-0.1), b"alpha must be finite and >= 0"), (dict(alpha=nan), b"alpha"),
             (dict(alpha=inf), b"alpha"), (dict(eps=0.0), b"eps must be finite and > 0"), (dict(eps=-1e-6), b"eps"),
             (dict(eps=nan), b"eps"), (dict(eps=inf), b"eps")]
    if td_f64:
        cases.append((dict(td=A64 + 4), b"aligned"))     # 4-byte aligned is not enough for fp64 errors
    for kw, msg in cases:
        args = dict(td_f64=td_f64)
        args.update(kw)
        assert _update(lib, t, **args) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and b"fg_per_update" in err, (msg, err)


SAMPLE_ARGS = ("u", "B", "beta", "done", "actions", "reward", "N", "A", "rows", "index", "stamp_out", "slot_out",
               "env_out", "done_out", "weights", "actions_out", "reward_out")


def _sample(lib, sfx, t, **kw):
    args = dict(B=64, beta=0.4, N=9, A=2, done=BASE + (20 << 12) + 1)
    for i, k in enumerate(SAMPLE_ARGS):
        args.setdefault(k, A64 + ((i + 1) << 16))
    args.update(kw)
    return getattr(lib, "fg_per_sample" + sfx)(C.byref(t) if t is not None else None,
                                               *[args[k] for k in SAMPLE_ARGS], None)


@pytest.mark.parametrize("sfx,item", [("", 4), ("_f64", 8)], ids=["f32", "f64"])
def test_sample_rejections(sfx, item):
    nat, lib = _lib()
    who = b"fg_per_sample" + sfx.encode()
    for t, msg in _tree_cases(nat):
        assert _sample(lib, sfx, t) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and who in err, (msg, err)
    t = _tree(nat)
    cases = [(dict(B=0), b"B must be >= 1"), (dict(B=-1), b"B must be >= 1"),
             (dict(N=0), b"N must be in [1, FG_MAX_AGENTS"), (dict(N=257), b"N must be in"),
             (dict(A=0), b"A must be in [1, 64]"), (dict(A=65), b"A must be in"),
             (dict(beta=-0.5), b"beta must be finite and >= 0"), (dict(beta=math.nan), b"beta"),
             (dict(beta=math.inf), b"beta")]
    for k in ("u", "done", "actions", "reward"):
        cases.append((dict(**{k: None}), b"u / done / actions / reward must be non-null"))
    for k in SAMPLE_ARGS[8:]:
        cases.append((dict(**{k: None}), b"outputs must be non-null"))
    for k in ("u", "rows", "index", "stamp_out", "slot_out", "env_out"):
        cases.append((dict(**{k: A64 + 4}), b"8-byte aligned"))
    for k in ("actions", "reward", "weights", "actions_out", "reward_out"):
        cases.append((dict(**{k: A64 + item // 2}), b"aligned to the real type"))
    for kw, msg in cases:
        assert _sample(lib, sfx, t, **kw) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and who in err, (msg, err)


# ------------------------------------------------------------------ Python layer
def _shell(dtype=torch.float32):
    from formation_gym import _native as nat
    from formation_gym.batched import SCENARIOS as SCN, BatchedFormationEnv, obs_dim
    env = BatchedFormationEnv.__new__(BatchedFormationEnv)
    env.scenario, env.scn, env.N, env.silent, env.dtype = "formation_hd_env", SCN["formation_hd_env"], 9, True, dtype
    env.L, env.E, env.act_dim = 9, 16, 2
    env.D = obs_dim(env.scenario, env.N, env.L)
    env.device = torch.device("cuda", 0)
    env.record_final = True
    assert env.scn == nat.FG_SCENARIO_HD
    return env


def test_alpha_and_eps_are_checked_first():
    from formation_gym import PrioritizedStateReplayBuffer
    env = _shell()
    for a in (-0.1, math.nan, math.inf):
        with pytest.raises(ValueError, match="alpha must be finite and >= 0"):
            PrioritizedStateReplayBuffer(env, 8, alpha=a)
    for e in (0.0, -1e-6, math.nan, math.inf):
        with pytest.raises(ValueError, match="eps must be finite and > 0"):
            PrioritizedStateReplayBuffer(env, 8, eps=e)
    env.record_final = False                              # the base class's checks still apply
    with pytest.raises(ValueError, match="record_final=True"):
        PrioritizedStateReplayBuffer(env, 8)


def _unbuilt(env):
    """A buffer object without device storage: what the argument checks read before any device call."""
    from formation_gym.replay import PrioritizedStateReplayBuffer
    buf = PrioritizedStateReplayBuffer.__new__(PrioritizedStateReplayBuffer)
    buf.env, buf.capacity, buf._valid = env, 8, {}
    return buf


def test_sample_errors_before_the_device():
    env = _shell()
    buf = _unbuilt(env)
    with pytest.raises(ValueError, match="no transition"):
        buf.sample(4)
    buf._valid = {1: 0}
    with pytest.raises(ValueError, match="batch_size"):
        buf.sample(0)
    for beta in (-0.1, math.nan, math.inf):
        with pytest.raises(ValueError, match="beta must be finite and >= 0"):
            buf.sample(4, beta)


def test_update_errors_before_the_device():
    from formation_gym.replay import _PrioritizedBatch
    env = _shell()
    buf, other = _unbuilt(env), _unbuilt(env)
    meta = torch.device("meta")
    ids = torch.zeros(2, 5, dtype=torch.int64, device=meta)

    def batch(owner, **kw):
        b = _PrioritizedBatch(index=ids[0], stamp=ids[1])
        b.update(kw)
        b.buffer = owner
        return b

    td = torch.zeros(5, device=meta)
    for b in (dict(index=ids[0], stamp=ids[1]), batch(other)):
        with pytest.raises(ValueError, match="sample\\(\\) result of this buffer"):
            buf.update_priorities(b, td)
    env.device = meta                                     # (a device tensor without a device)
    good = batch(buf)
    for b in (batch(buf, index=ids[0].int()), batch(buf, stamp=ids[1][:3]), batch(buf, index=None),
              batch(buf, index=torch.zeros(5, dtype=torch.int64))):
        with pytest.raises(ValueError, match="must be the int64 \\[B\\] device tensors"):
            buf.update_priorities(b, td)
    for bad in (torch.zeros(5, dtype=torch.float16, device=meta), torch.zeros(5, dtype=torch.int64, device=meta),
                [0.0] * 5):
        with pytest.raises(ValueError, match="float32 or float64"):
            buf.update_priorities(good, bad)
    for bad in (torch.zeros(4, device=meta), torch.zeros(5, 1, device=meta), torch.zeros(5, 9, device=meta)):
        with pytest.raises(ValueError, match="shape"):
            buf.update_priorities(good, bad)
    with pytest.raises(ValueError, match="must be on meta"):
        buf.update_priorities(good, torch.zeros(5, dtype=torch.float64))
