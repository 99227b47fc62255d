"""Target banks of formation_hd_env (include/formation_gym_b200.h fg_targets), CPU only: the *_targets entry points
reject bad banks before any device call, and BatchedFormationEnv validates a bank before it touches a device."""
import ctypes as C

import numpy as np
import pytest


def _lib():
    from formation_gym import _native as nat
    return nat, nat.load()


def _call(lib, nat, name, sfx, scenario, t, N=9):
    """One call of entry point `name` with empty buffers; the bank is checked first, so nothing else matters."""
    p, b = nat.make_params(), nat.fg_buffers()
    f = getattr(lib, name + sfx)
    if name == "fg_reset_targets":
        return f(C.byref(p), C.byref(b), scenario, 4, N, N, None, 0, 0, 0, None, C.byref(t))
    if name == "fg_step_fused_targets":
        return f(C.byref(p), C.byref(b), scenario, 4, N, N, 1, 0, 1, 0, 0, 0, None, C.byref(t))
    return f(C.byref(p), C.byref(b), scenario, 4, N, N, 1, 3, 1, 0, 0, 0, None, C.byref(t))


ENTRIES = ["fg_reset_targets", "fg_step_fused_targets", "fg_step_policy_targets"]


@pytest.mark.parametrize("sfx,item", [("", 8), ("_f64", 16)], ids=["f32", "f64"])
@pytest.mark.parametrize("name", ENTRIES)
def test_bad_target_banks_are_rejected_without_a_device(name, sfx, item):
    nat, lib = _lib()
    base = 1 << 20                                       # never dereferenced: validation happens first

    def bank(shapes=base, vels=None, index=None, count=2):
        t = nat.fg_targets()
        t.shapes, t.vels, t.index, t.count = shapes, vels, index, count
        return t

    cases = [
        (nat.FG_SCENARIO_BASIC, bank(), b"formation_hd_env only"),
        (nat.FG_SCENARIO_HD_PARTIAL, bank(), b"formation_hd_env only"),
        (nat.FG_SCENARIO_HD_PARTIAL_RANGE, bank(), b"formation_hd_env only"),
        (nat.FG_SCENARIO_HD_OBSTACLE, bank(), b"formation_hd_env only"),
        (nat.FG_SCENARIO_HD, bank(count=0), b"count must be >= 1"),
        (nat.FG_SCENARIO_HD, bank(count=-3), b"count must be >= 1"),
        (nat.FG_SCENARIO_HD, bank(shapes=None), b"shapes must be non-null"),
        (nat.FG_SCENARIO_HD, bank(shapes=base + item // 2), b"aligned"),
        (nat.FG_SCENARIO_HD, bank(vels=base + item // 2), b"aligned"),
        (nat.FG_SCENARIO_HD, bank(index=base + 2), b"aligned"),
    ]
    if item == 16:
        cases.append((nat.FG_SCENARIO_HD, bank(shapes=base + 8), b"aligned"))   # float2-aligned is not enough in fp64
    for scenario, t, msg in cases:
        rc = _call(lib, nat, name, sfx, scenario, t)
        assert rc == -1, (scenario, msg)          # FG_ERR_ARG
        assert msg in lib.fg_last_error(), (msg, lib.fg_last_error())


@pytest.mark.parametrize("name", ENTRIES)
def test_valid_bank_reaches_the_ordinary_checks(name):
    """A well-formed bank passes its own checks; the call then fails on the (empty) buffers like the plain entry
    point -- still without a device."""
    nat, lib = _lib()
    t = nat.fg_targets()
    t.shapes, t.vels, t.index, t.count = 1 << 20, 1 << 21, 1 << 22, 7
    rc = _call(lib, nat, name, "", nat.FG_SCENARIO_HD, t)
    assert rc == -1 and b"fg_targets" not in lib.fg_last_error()
    assert b"non-null" in lib.fg_last_error()


def _env(**kw):
    from formation_gym.batched import BatchedFormationEnv
    args = dict(scenario="formation_hd_env", num_envs=6, num_agents=9)
    args.update(kw)
    return BatchedFormationEnv(**args)


def test_python_bank_validation_errors():
    """BatchedFormationEnv checks a bank before it loads the library or looks for a device."""
    shapes = np.zeros((3, 9, 2))
    with pytest.raises(ValueError, match="formation_hd_env only"):
        _env(scenario="basic_formation_env", num_agents=3, target_shapes=np.zeros((3, 3, 2)))
    for scn in ("formation_hd_partial_env", "formation_hd_partial_range_env", "formation_hd_obs_env"):
        with pytest.raises(ValueError, match="formation_hd_env only"):
            _env(scenario=scn, num_agents=4, target_shapes=np.zeros((3, 4, 2)))
    with pytest.raises(ValueError, match=r"target_shapes must have shape \(K, 9, 2\)"):
        _env(target_shapes=np.zeros((3, 8, 2)))
    with pytest.raises(ValueError, match=r"target_shapes must have shape"):
        _env(target_shapes=np.zeros((9, 2)))
    with pytest.raises(ValueError, match=r"K >= 1"):
        _env(target_shapes=np.zeros((0, 9, 2)))
    with pytest.raises(ValueError, match=r"target_vels must have shape \(3, 2\)"):
        _env(target_shapes=shapes, target_vels=np.zeros((2, 2)))
    with pytest.raises(ValueError, match=r"target_vels must have shape \(3, 2\)"):
        _env(target_shapes=shapes, target_vels=np.zeros(2))
    with pytest.raises(ValueError, match=r"target_index must have shape \(6,\)"):
        _env(target_shapes=shapes, target_index=np.zeros(5, np.int64))
    with pytest.raises(ValueError, match="integers"):
        _env(target_shapes=shapes, target_index=np.zeros(6))
    with pytest.raises(ValueError, match="need target_shapes"):
        _env(target_vels=np.zeros((3, 2)))
    with pytest.raises(ValueError, match="need target_shapes"):
        _env(target_index=np.zeros(6, np.int32))


def test_bank_index_conversion_keeps_out_of_range_out_of_range():
    """Indices beyond int32 must not wrap into a valid task when they are narrowed."""
    from formation_gym.batched import _target_bank
    shapes, vels, index = _target_bank("formation_hd_env", 4, 3, np.zeros((2, 3, 2)), None,
                                       np.array([0, 1, 2 ** 32, -2 ** 40]))
    assert vels is None and tuple(shapes.shape) == (2, 3, 2)
    assert index.tolist() == [0, 1, 2 ** 31 - 1, -1]
    assert _target_bank("formation_hd_env", 4, 3, None, None, None) is None


def test_sharded_env_checks_the_job_index_shape():
    from formation_gym import distributed as fgd
    with pytest.raises(ValueError, match=r"target_index must have shape \(10,\)"):
        fgd.make_sharded_env("formation_hd_env", 10, 3, target_shapes=np.zeros((2, 3, 2)), target_index=np.zeros(4))
