"""State-record replay (include/formation_gym_b200.h fg_obs_gather, formation_gym.replay), CPU only: fg_obs_gather rejects
bad arguments before any device call, and the Python layer rejects what it cannot decode before it touches a device."""
import ctypes as C

import pytest
import torch

BASE = 1 << 20                                           # never dereferenced: validation happens first
SCENARIOS = ["HD", "BASIC", "HD_PARTIAL", "HD_PARTIAL_RANGE", "HD_OBSTACLE"]


def _lib():
    from formation_gym import _native as nat
    return nat, nat.load()


def _block(nat, scenario, silent=True, **kw):
    """A well-formed state block for `scenario` (distinct aligned addresses), then the overrides."""
    f = nat.fg_final()
    f.pos, f.vel = BASE, BASE + (1 << 12)
    if not silent:
        f.comm = BASE + (2 << 12)
    if scenario == nat.FG_SCENARIO_HD:
        f.ideal_shape, f.ideal_vel = BASE + (3 << 12), BASE + (4 << 12)
    else:
        f.landmarks = BASE + (5 << 12)
    for k, v in kw.items():
        setattr(f, k, v)
    return f


def _gather(lib, nat, sfx, scenario, f, R=100, rows=BASE + (6 << 12), B=8, obs=BASE + (7 << 12), silent=True, N=None,
            L=None):
    p = nat.make_params(silent=silent)
    N = N if N is not None else (9 if scenario == nat.FG_SCENARIO_HD else 4)
    L = L if L is not None else (N if scenario in (nat.FG_SCENARIO_HD, nat.FG_SCENARIO_BASIC) else 7)
    fb = C.byref(f) if f is not None else None
    return getattr(lib, "fg_obs_gather" + sfx)(C.byref(p), fb, R, rows, B, obs, scenario, N, L, None)


def _cases(nat, item, scenario):
    hd = scenario == nat.FG_SCENARIO_HD
    cases = [
        (_block(nat, scenario, pos=None), {}, b"pos / vel must be non-null"),
        (_block(nat, scenario, vel=None), {}, b"pos / vel must be non-null"),
        (_block(nat, scenario, pos=BASE + item // 2), {}, b"aligned"),
        (_block(nat, scenario, vel=BASE + item // 2), {}, b"aligned"),
    ]
    if hd:
        cases += [(_block(nat, scenario, ideal_shape=None), {}, b"ideal_shape / ideal_vel must be non-null"),
                  (_block(nat, scenario, ideal_vel=None), {}, b"ideal_shape / ideal_vel must be non-null"),
                  (_block(nat, scenario, ideal_shape=BASE + item // 2), {}, b"aligned"),
                  (_block(nat, scenario, ideal_vel=BASE + item // 2), {}, b"aligned")]
    else:
        cases += [(_block(nat, scenario, landmarks=None), {}, b"landmarks must be non-null"),
                  (_block(nat, scenario, landmarks=BASE + item // 2), {}, b"aligned")]
    if scenario != nat.FG_SCENARIO_HD_OBSTACLE:                # (formation_hd_obs_env has silent agents only)
        cases += [(_block(nat, scenario, silent=False, comm=None), dict(silent=False), b"comm must be non-null"),
                  (_block(nat, scenario, silent=False, comm=BASE + item // 2), dict(silent=False), b"aligned")]
    if item == 16:                                             # float2-aligned is not enough in fp64
        cases.append((_block(nat, scenario, pos=BASE + 8), {}, b"aligned"))
    return cases


@pytest.mark.parametrize("sfx,item", [("", 8), ("_f64", 16)], ids=["f32", "f64"])
@pytest.mark.parametrize("scn", SCENARIOS)
def test_bad_state_blocks_are_rejected_without_a_device(scn, sfx, item):
    nat, lib = _lib()
    scenario = getattr(nat, "FG_SCENARIO_" + scn)
    for f, kw, msg in _cases(nat, item, scenario):
        assert _gather(lib, nat, sfx, scenario, f, **kw) == -1, msg           # FG_ERR_ARG
        err = lib.fg_last_error()
        assert msg in err and b"fg_obs_gather" in err, (msg, err)


@pytest.mark.parametrize("sfx", ["", "_f64"], ids=["f32", "f64"])
@pytest.mark.parametrize("scn", SCENARIOS)
def test_bad_gather_arguments_are_rejected_without_a_device(scn, sfx):
    nat, lib = _lib()
    scenario = getattr(nat, "FG_SCENARIO_" + scn)
    f = _block(nat, scenario)
    cases = [(dict(f=None), b"state block must be non-null"),
             (dict(rows=None), b"rows / obs must be non-null"),
             (dict(obs=None), b"rows / obs must be non-null"),
             (dict(R=0), b"R and B must be >= 1"),
             (dict(R=-(1 << 40)), b"R and B must be >= 1"),
             (dict(B=0), b"R and B must be >= 1"),
             (dict(B=-3), b"R and B must be >= 1"),
             (dict(rows=BASE + 4), b"rows must be 8-byte aligned")]
    for kw, msg in cases:
        args = dict(f=f)
        args.update(kw)
        assert _gather(lib, nat, sfx, scenario, args.pop("f"), **args) == -1, msg
        err = lib.fg_last_error()
        assert msg in err and b"fg_obs_gather" in err, (msg, err)


@pytest.mark.parametrize("sfx", ["", "_f64"], ids=["f32", "f64"])
def test_valid_gather_reaches_the_ordinary_checks(sfx):
    """A well-formed call goes on to the ordinary argument checks (an unknown scenario id; E*N = B*N too large) --
    still without a device.  A record count past 2^32 is accepted (64-bit addressing)."""
    nat, lib = _lib()
    f = _block(nat, nat.FG_SCENARIO_HD, landmarks=BASE + (5 << 12))
    assert _gather(lib, nat, sfx, 17, f, R=1 << 40) == -1
    assert b"unknown scenario" in lib.fg_last_error()
    assert _gather(lib, nat, sfx, nat.FG_SCENARIO_HD, f, R=1 << 40, B=1 << 30) == -1
    assert b"E*N must be < 2^31" in lib.fg_last_error()


class _Shell:
    """The attributes BatchedFormationEnv.gather_observations reads, without a device."""


def _shell(scenario="formation_hd_env", N=9, L=None, silent=True, dtype=torch.float32):
    from formation_gym import _native as nat
    from formation_gym.batched import SCENARIOS as SCN, BatchedFormationEnv, obs_dim
    env = BatchedFormationEnv.__new__(BatchedFormationEnv)
    env.scenario, env.scn, env.N, env.silent, env.dtype = scenario, SCN[scenario], N, silent, dtype
    env.L = N if env.scn == nat.FG_SCENARIO_HD else (L or 4)
    env.D = obs_dim(scenario, N, env.L)
    env.device = torch.device("cuda", 0)
    return env


def _states(env, R=5, dtype=None, device="cpu"):
    dtype = dtype or env.dtype
    shapes = {"ideal_vel": (R, 2), "landmarks": (R, env.L, 2)}
    return {k: torch.zeros(*shapes.get(k, (R, env.N, 2)), dtype=dtype, device=device) for k in env.state_record_keys()}


@pytest.mark.parametrize("scenario", ["formation_hd_env", "basic_formation_env", "formation_hd_obs_env"])
def test_gather_observations_checks_before_the_device(scenario):
    env = _shell(scenario)
    rows = torch.zeros(4, dtype=torch.int64)
    keys = env.state_record_keys()
    for k in keys:                                          # missing array, wrong dtype, wrong shape
        st = _states(env)
        del st[k]
        with pytest.raises(ValueError, match="must be a tensor"):
            env.gather_observations(st, rows)
        st = _states(env)
        st[k] = st[k].double()
        with pytest.raises(ValueError, match="dtype"):
            env.gather_observations(st, rows)
        st = _states(env)
        st[k] = torch.zeros(*st[k].shape[:-1], 3)
        with pytest.raises(ValueError, match="shape"):
            env.gather_observations(st, rows)
    st = _states(env)
    st[keys[-1]] = torch.zeros(6, *st[keys[-1]].shape[1:])  # record counts disagree
    with pytest.raises(ValueError, match="shape"):
        env.gather_observations(st, rows)
    with pytest.raises(ValueError, match="at least one record"):
        env.gather_observations(_states(env, R=0), rows)
    for bad in (rows.int(), rows.float(), rows[None], rows[:0], [0, 1]):
        with pytest.raises(ValueError, match="rows must be a non-empty 1-D int64"):
            env.gather_observations(_states(env), bad)
    for bad in (torch.zeros(4, env.N, env.D + 1), torch.zeros(4, env.N, env.D, dtype=torch.float64),
                torch.zeros(3, env.N, env.D)):
        with pytest.raises(ValueError, match="out must be"):
            env.gather_observations(_states(env), rows, out=bad)
    with pytest.raises(ValueError, match="must be on cuda:0"):   # everything else right, but on the host
        env.gather_observations(_states(env), rows)


def test_gather_observations_needs_comm_for_non_silent_agents():
    env = _shell(silent=False)
    assert "comm" in env.state_record_keys()
    st = _states(env)
    del st["comm"]
    with pytest.raises(ValueError, match="comm"):
        env.gather_observations(st, torch.zeros(2, dtype=torch.int64))


def test_replay_buffer_needs_record_final_and_two_slots():
    from formation_gym import StateReplayBuffer
    env = _shell()
    env.record_final = False
    with pytest.raises(ValueError, match="record_final=True"):
        StateReplayBuffer(env, 8)
    env.record_final = True
    for cap in (1, 0, -4):
        with pytest.raises(ValueError, match="capacity must be >= 2"):
            StateReplayBuffer(env, cap)
