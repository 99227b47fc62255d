"""Terminal blocks (include/formation_gym_b200.h fg_final), CPU only: the *_final entry points and fg_final_obs reject
bad blocks before any device call, and BatchedFormationEnv rejects what a terminal block cannot record before it
touches a device."""
import ctypes as C

import pytest


def _lib():
    from formation_gym import _native as nat
    return nat, nat.load()


BASE = 1 << 20                                           # never dereferenced: validation happens first


def _call(lib, nat, name, sfx, scenario, f, N=9, L=9, silent=True, auto_reset=1, n_steps=1, t=None):
    """One call of entry point `name` with empty buffers; the terminal block is checked first."""
    p, b = nat.make_params(silent=silent), nat.fg_buffers()
    fn = getattr(lib, name + sfx)
    tb = C.byref(t) if t is not None else None
    if name == "fg_final_obs":
        return fn(C.byref(p), C.byref(f), BASE, BASE, scenario, 4, N, L, None)
    if name == "fg_step_fused_final":
        return fn(C.byref(p), C.byref(b), scenario, 4, N, L, n_steps, 1, auto_reset, 0, 0, 0, None, tb, C.byref(f))
    return fn(C.byref(p), C.byref(b), scenario, 4, N, L, n_steps, 3, auto_reset, 0, 0, 0, None, tb, C.byref(f))


def _block(nat, scenario, silent=True, **kw):
    """A well-formed terminal block for `scenario` (distinct aligned addresses), then the overrides."""
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


STEPS = ["fg_step_fused_final", "fg_step_policy_final"]
SCENARIOS = ["HD", "BASIC", "HD_PARTIAL", "HD_PARTIAL_RANGE", "HD_OBSTACLE"]


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
@pytest.mark.parametrize("name", STEPS + ["fg_final_obs"])
def test_bad_terminal_blocks_are_rejected_without_a_device(name, scn, sfx, item):
    nat, lib = _lib()
    scenario = getattr(nat, "FG_SCENARIO_" + scn)
    N = 9 if scenario == nat.FG_SCENARIO_HD else 4
    L = N if scenario in (nat.FG_SCENARIO_HD, nat.FG_SCENARIO_BASIC) else 7
    for f, kw, msg in _cases(nat, item, scenario):
        rc = _call(lib, nat, name, sfx, scenario, f, N=N, L=L, **kw)
        assert rc == -1, msg                                   # FG_ERR_ARG
        assert msg in lib.fg_last_error(), (msg, lib.fg_last_error())
        assert b"fg_final" in lib.fg_last_error()


@pytest.mark.parametrize("sfx", ["", "_f64"], ids=["f32", "f64"])
@pytest.mark.parametrize("name", STEPS)
def test_steps_with_a_block_need_one_auto_resetting_step(name, sfx):
    nat, lib = _lib()
    f = _block(nat, nat.FG_SCENARIO_HD)
    rc = _call(lib, nat, name, sfx, nat.FG_SCENARIO_HD, f, auto_reset=0)
    assert rc == -1 and b"needs auto_reset != 0" in lib.fg_last_error()
    for n in (0, 2, 25):
        rc = _call(lib, nat, name, sfx, nat.FG_SCENARIO_HD, f, n_steps=n)
        assert rc == -1 and b"needs n_steps == 1" in lib.fg_last_error()


@pytest.mark.parametrize("sfx", ["", "_f64"], ids=["f32", "f64"])
@pytest.mark.parametrize("name", STEPS)
def test_bank_checks_stay_with_a_block(name, sfx):
    """The target-bank checks of the _targets calls apply unchanged to the _final calls."""
    nat, lib = _lib()
    t = nat.fg_targets()
    t.shapes, t.count = BASE, 0
    rc = _call(lib, nat, name, sfx, nat.FG_SCENARIO_HD, _block(nat, nat.FG_SCENARIO_HD), t=t)
    assert rc == -1 and b"count must be >= 1" in lib.fg_last_error()


def test_final_obs_needs_a_block_done_and_obs():
    nat, lib = _lib()
    p = nat.make_params()
    for sfx in ("", "_f64"):
        fn = getattr(lib, "fg_final_obs" + sfx)
        assert fn(C.byref(p), None, BASE, BASE, nat.FG_SCENARIO_HD, 4, 9, 9, None) == -1
        assert b"terminal block must be non-null" in lib.fg_last_error()
        f = _block(nat, nat.FG_SCENARIO_HD)
        assert fn(C.byref(p), C.byref(f), None, BASE, nat.FG_SCENARIO_HD, 4, 9, 9, None) == -1
        assert b"done / obs must be non-null" in lib.fg_last_error()
        assert fn(C.byref(p), C.byref(f), BASE, None, nat.FG_SCENARIO_HD, 4, 9, 9, None) == -1
        assert b"done / obs must be non-null" in lib.fg_last_error()


@pytest.mark.parametrize("scn", SCENARIOS)
@pytest.mark.parametrize("name", STEPS)
def test_valid_block_reaches_the_ordinary_checks(name, scn):
    """A well-formed block (with or without a bank) passes its own checks; the call then fails on the (empty) buffers
    like the plain entry point -- still without a device."""
    nat, lib = _lib()
    scenario = getattr(nat, "FG_SCENARIO_" + scn)
    N = 9 if scenario == nat.FG_SCENARIO_HD else 4
    L = N if scenario in (nat.FG_SCENARIO_HD, nat.FG_SCENARIO_BASIC) else 7
    banks = [None]
    if scenario == nat.FG_SCENARIO_HD:
        t = nat.fg_targets()
        t.shapes, t.vels, t.index, t.count = 1 << 24, 1 << 25, 1 << 26, 3
        banks.append(t)
    for t in banks:
        rc = _call(lib, nat, name, "", scenario, _block(nat, scenario), N=N, L=L, t=t)
        assert rc == -1
        err = lib.fg_last_error()
        assert b"fg_final" not in err and b"fg_targets" not in err, err


def test_valid_block_reaches_the_final_obs_arguments():
    """fg_final_obs with a valid block goes on to the ordinary argument checks (here: an unknown scenario id)."""
    nat, lib = _lib()
    p = nat.make_params()
    f = _block(nat, nat.FG_SCENARIO_HD, landmarks=BASE + (5 << 12))
    assert lib.fg_final_obs(C.byref(p), C.byref(f), BASE, BASE, 17, 4, 9, 9, None) == -1
    assert b"unknown scenario" in lib.fg_last_error()


def _env(**kw):
    from formation_gym.batched import BatchedFormationEnv
    args = dict(scenario="formation_hd_env", num_envs=6, num_agents=9)
    args.update(kw)
    return BatchedFormationEnv(**args)


def test_python_record_final_needs_auto_reset():
    """BatchedFormationEnv / CudaVecEnv reject record_final without auto-reset before they look for a device."""
    with pytest.raises(ValueError, match="needs auto_reset=True"):
        _env(record_final=True, auto_reset=False)
    from formation_gym.vec_env import make_vec_env
    with pytest.raises(ValueError, match="needs auto_reset=True"):
        make_vec_env("formation_hd_env", 4, 9, record_final=True, auto_reset=False)


def test_python_multi_step_calls_are_rejected_with_a_block():
    """rollout_random(n > 1) and step_bfs(n_steps > 1) are refused before any launch; final_observation needs a
    block.  (An object without device buffers: the checks come before anything that would touch them.)"""
    from formation_gym import _native as nat
    from formation_gym.batched import BatchedFormationEnv
    env = BatchedFormationEnv.__new__(BatchedFormationEnv)
    env._final = nat.fg_final()
    with pytest.raises(ValueError, match="one step per call"):
        env.rollout_random(2)
    with pytest.raises(ValueError, match="one step per call"):
        env.step_bfs(3, n_steps=2)
    env._final = None
    with pytest.raises(ValueError, match="needs record_final=True"):
        env.final_observation()
