"""On-policy rollout storage (include/formation_gym_b200.h fg_gae, formation_gym.rollout.StateRolloutBuffer), CPU only:
every argument rejection of fg_gae / fg_gae_f64 before any device call, and the Python errors the buffer raises before
it touches a device."""
import math

import pytest
import torch

BASE = 1 << 20                                           # never dereferenced: validation happens first
ARGS = ("reward", "value", "final_value", "done", "adv", "ret", "T", "E", "N", "gamma", "lam")


def _lib():
    from formation_gym import _native as nat
    return nat, nat.load()


def _gae(lib, sfx, **kw):
    args = dict(reward=BASE + (1 << 16), value=BASE + (2 << 16), final_value=BASE + (3 << 16),
                done=BASE + (4 << 16) + 1, adv=BASE + (5 << 16), ret=BASE + (6 << 16), T=25, E=1024, N=9,
                gamma=0.99, lam=0.95)
    args.update(kw)
    return getattr(lib, "fg_gae" + sfx)(*[args[k] for k in ARGS], None)


@pytest.mark.parametrize("sfx,item", [("", 4), ("_f64", 8)], ids=["f32", "f64"])
def test_gae_rejections(sfx, item):
    nat, lib = _lib()
    who = b"fg_gae" + sfx.encode()
    inf, nan = math.inf, math.nan
    cases = []
    for k in ("reward", "value", "done", "adv", "ret"):
        cases.append((dict(**{k: None}), b"reward / value / done / adv / ret must be non-null"))
    cases += [(dict(T=0), b"T must be >= 1"), (dict(T=-3), b"T must be >= 1"),
              (dict(E=0), b"E must be >= 1"), (dict(E=-1), b"E must be >= 1"),
              (dict(N=0), b"N must be in [1, FG_MAX_AGENTS"), (dict(N=257), b"N must be in"),
              (dict(T=1, E=(1 << 48) // 9 + 1, N=9), b"T * E * N must be <= 2^48"),
              (dict(T=1 << 20, E=(1 << 20) + 1, N=256), b"<= 2^48"), (dict(T=(1 << 31) - 1, E=1 << 40, N=256), b"<= 2^48")]
    for name, key in (("gamma", "gamma"), ("lambda", "lam")):
        for bad in (-0.01, 1.0 + 1e-12, nan, inf, -inf):
            cases.append((dict(**{key: bad}), (name + " must be finite and in [0, 1]").encode()))
    for k in ("reward", "value", "final_value", "adv", "ret"):
        cases.append((dict(**{k: BASE + (7 << 16) + item // 2}), b"must be aligned to the real type"))
        if item == 8:                                    # 4-byte aligned is not enough for fp64
            cases.append((dict(**{k: BASE + (7 << 16) + 4}), b"aligned to the real type"))
    for kw, msg in cases:
        assert _gae(lib, sfx, **kw) == -1, (kw, msg)
        err = lib.fg_last_error()
        assert msg in err and who in err, (kw, msg, err)


# ------------------------------------------------------------------ Python layer
def _shell(dtype=torch.float32):
    """A device-less formation_hd_env (N = 9, E = 16) whose tensors live on the meta device."""
    from formation_gym import _native as nat
    from formation_gym.batched import SCENARIOS as SCN, BatchedFormationEnv, obs_dim
    env = BatchedFormationEnv.__new__(BatchedFormationEnv)
    env.scenario, env.scn, env.N, env.silent, env.dtype = "formation_hd_env", SCN["formation_hd_env"], 9, True, dtype
    env.L, env.E, env.act_dim = 9, 16, 2
    env.D = obs_dim(env.scenario, env.N, env.L)
    env.device = torch.device("meta")
    env.auto_reset = True
    assert env.scn == nat.FG_SCENARIO_HD
    return env


def _buffer(env, T=4):
    from formation_gym import StateRolloutBuffer
    return StateRolloutBuffer(env, T)


def test_constructor_errors():
    from formation_gym import StateRolloutBuffer
    env = _shell()
    for T in (0, -1):
        with pytest.raises(ValueError, match="num_steps must be >= 1"):
            StateRolloutBuffer(env, T)
    env.auto_reset = False
    with pytest.raises(ValueError, match="auto_reset=True"):
        StateRolloutBuffer(env, 4)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_storage_shapes(dtype):
    env = _shell(dtype)
    buf = _buffer(env, 5)
    E, N = env.E, env.N
    assert set(buf.states) == {"pos", "vel", "ideal_shape", "ideal_vel"}
    assert buf.states["pos"].shape == (5 * E, N, 2) and buf.states["ideal_vel"].shape == (5 * E, 2)
    assert buf.actions.shape == (5, E, N, 2) and buf.values.shape == (6, E, N) and buf.done.shape == (5, E)
    for k in ("log_probs", "rewards", "advantages", "returns"):
        assert getattr(buf, k).shape == (5, E, N) and getattr(buf, k).dtype == dtype
    assert buf.done.dtype == torch.bool and buf.final_values is None and buf.step == -1


def test_insert_errors_before_the_device():
    env = _shell()
    buf = _buffer(env, 4)
    meta = torch.device("meta")
    E, N = env.E, env.N
    act, lp, v = torch.zeros(E, N, 2, device=meta), torch.zeros(E, N, device=meta), torch.zeros(E, N, device=meta)
    with pytest.raises(ValueError, match="call start\\(\\)"):
        buf.insert(act, lp, v)
    buf._t = 0                                           # (as start() leaves it)
    bad_shapes = [(dict(actions=torch.zeros(E, N, 4, device=meta)), "actions must have shape"),
                  (dict(actions=torch.zeros(E, N, device=meta)), "actions must have shape"),
                  (dict(log_probs=torch.zeros(E, N, 1, device=meta)), "log_probs must have shape"),
                  (dict(values=torch.zeros(E, device=meta)), "values must have shape"),
                  (dict(values=torch.zeros(N, E, device=meta)), "values must have shape"),
                  (dict(final_values=torch.zeros(E, N, 2, device=meta)), "final_values must have shape")]
    bad_types = [(dict(actions=torch.zeros(E, N, 2, dtype=torch.int64, device=meta)), "actions must be a floating"),
                 (dict(log_probs=torch.zeros(E, N, dtype=torch.bool, device=meta)), "log_probs must be a floating"),
                 (dict(values=torch.zeros(E, N, dtype=torch.int32, device=meta)), "values must be a floating"),
                 (dict(final_values=torch.zeros(E, N, dtype=torch.uint8, device=meta)), "final_values must be a float"),
                 (dict(values=[[0.0] * N] * E), "values must be a tensor")]
    host = [(dict(actions=torch.zeros(E, N, 2)), "actions must be on meta"),
            (dict(log_probs=torch.zeros(E, N)), "log_probs must be on meta"),
            (dict(values=torch.zeros(E, N, dtype=torch.float64)), "values must be on meta"),
            (dict(final_values=torch.zeros(E, N)), "final_values must be on meta")]
    for kw, msg in bad_shapes + bad_types + host:
        args = dict(actions=act, log_probs=lp, values=v)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            buf.insert(**args)
        assert buf.step == 0                             # nothing recorded
    buf._t = 4
    with pytest.raises(ValueError, match="already holds num_steps = 4 steps"):
        buf.insert(act, lp, v)


def test_compute_returns_errors_before_the_device():
    env = _shell()
    buf = _buffer(env, 4)
    nv = torch.zeros(env.E, env.N, device=torch.device("meta"))
    for t in (-1, 0, 3):
        buf._t = t
        with pytest.raises(ValueError, match="needs num_steps = 4 inserts since start\\(\\), got %d" % max(t, 0)):
            buf.compute_returns(nv)
    buf._t = 4
    for kw, msg in ((dict(gamma=1.5), "gamma must be finite"), (dict(gamma=math.nan), "gamma must be finite"),
                    (dict(gamma=-0.1), "gamma"), (dict(gae_lambda=-0.5), "gae_lambda must be finite"),
                    (dict(gae_lambda=math.inf), "gae_lambda")):
        with pytest.raises(ValueError, match=msg):
            buf.compute_returns(nv, **kw)
    for bad, msg in ((torch.zeros(env.E, device=torch.device("meta")), "next_values must have shape"),
                     (torch.zeros(env.E, env.N, dtype=torch.int64, device=torch.device("meta")), "floating"),
                     (torch.zeros(env.E, env.N), "next_values must be on meta")):
        with pytest.raises(ValueError, match=msg):
            buf.compute_returns(bad)


def test_minibatches_errors_before_the_device():
    env = _shell()
    buf = _buffer(env, 4)
    with pytest.raises(ValueError, match="call compute_returns\\(\\)"):
        buf.minibatches(2)
    buf._t, buf._ready = 3, False                        # (an insert after compute_returns also clears it)
    with pytest.raises(ValueError, match="call compute_returns\\(\\)"):
        buf.minibatches(2)
    buf._t, buf._ready = 4, True
    for n in (0, -1, 4 * env.E + 1):
        with pytest.raises(ValueError, match="num_mini_batch must be in \\[1, T\\*E = 64\\]"):
            buf.minibatches(n)
