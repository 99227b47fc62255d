"""ctypes binding of include/formation_gym_b200.h (the C ABI of the sm_100a kernels).

There is NO CPU fallback: if the shared library is missing or a call fails this module raises.
Pointers are raw device addresses (``tensor.data_ptr()``); the stream is the caller's CUDA stream.
"""
import ctypes as C
import os

from . import _build

FG_ABI_VERSION = 9
FG_MAX_AGENTS = 256
FG_MAX_LANDMARKS = 256
FG_MAX_WALLS = 8
FG_SCENARIO_HD = 0
FG_SCENARIO_BASIC = 1
FG_SCENARIO_HD_PARTIAL = 2
FG_SCENARIO_HD_PARTIAL_RANGE = 3
FG_SCENARIO_HD_OBSTACLE = 4

EXPORTS = [
    "fg_abi_version", "fg_last_error", "fg_device_info", "fg_launch_geometry", "fg_set_option", "fg_get_option",
    "fg_world_step", "fg_world_step_f64", "fg_obs_reward", "fg_obs_reward_f64",
    "fg_step_fused", "fg_step_fused_f64", "fg_reset", "fg_reset_f64",
    "fg_random_actions", "fg_random_actions_f64", "fg_fp32_probe", "fg_write_probe", "fg_policy_bfs", "fg_policy_bfs_f64",
    "fg_obs_to_host", "fg_pair_distances", "fg_pair_distances_f64", "fg_step_policy", "fg_step_policy_f64",
    "fg_reset_targets", "fg_reset_targets_f64", "fg_step_fused_targets", "fg_step_fused_targets_f64",
    "fg_step_policy_targets", "fg_step_policy_targets_f64", "fg_step_fused_final", "fg_step_fused_final_f64",
    "fg_step_policy_final", "fg_step_policy_final_f64", "fg_final_obs", "fg_final_obs_f64",
    "fg_obs_gather", "fg_obs_gather_f64", "fg_per_layout", "fg_per_fill", "fg_per_update", "fg_per_sample",
    "fg_per_sample_f64", "fg_gae", "fg_gae_f64",
]


class NativeError(RuntimeError):
    pass


class fg_wall(C.Structure):
    _fields_ = [("orient", C.c_int32), ("hard", C.c_int32), ("axis_pos", C.c_double),
                ("end0", C.c_double), ("end1", C.c_double), ("width", C.c_double)]


class fg_params(C.Structure):
    _fields_ = [
        ("dt", C.c_double), ("damping", C.c_double), ("contact_force", C.c_double),
        ("contact_margin", C.c_double), ("sensitivity", C.c_double), ("agent_size", C.c_double),
        ("mass", C.c_double), ("accel", C.c_double), ("max_speed", C.c_double),
        ("u_noise", C.c_double), ("c_noise", C.c_double), ("obs_range", C.c_double),
        ("obstacle_size", C.c_double), ("obstacle_mass", C.c_double), ("obstacle_floor", C.c_double),
        ("obstacle_fall_vy", C.c_double),
        ("has_accel", C.c_int32), ("has_max_speed", C.c_int32), ("collide", C.c_int32),
        ("silent", C.c_int32), ("world_length", C.c_int32), ("n_walls", C.c_int32),
        ("action_prescaled", C.c_int32), ("num_obs", C.c_int32), ("num_obstacles", C.c_int32),
        ("num_landmarks", C.c_int32),
        ("agent_mass", C.c_void_p), ("agent_size_arr", C.c_void_p),
        ("agent_accel", C.c_void_p), ("agent_max_speed", C.c_void_p),
        ("walls", fg_wall * FG_MAX_WALLS),
    ]


class fg_buffers(C.Structure):
    _fields_ = [
        ("pos", C.c_void_p), ("vel", C.c_void_p), ("act", C.c_void_p), ("comm", C.c_void_p),
        ("ideal_shape", C.c_void_p), ("ideal_vel", C.c_void_p), ("landmarks", C.c_void_p),
        ("step", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p), ("indiv", C.c_void_p),
        ("done", C.c_void_p), ("ep_return", C.c_void_p), ("ep_collisions", C.c_void_p),
        ("stats", C.c_void_p), ("landmark_vel", C.c_void_p), ("tick_dev", C.c_void_p),
        ("contact_pos", C.c_void_p), ("nan_flag", C.c_void_p),
    ]


class fg_targets(C.Structure):
    """Target bank of formation_hd_env (the ``*_targets`` entry points): K raw shapes [K,N,2], optional ideal
    velocities [K,2] and an optional per-env task index [E] (out of [0, K) = draw)."""
    _fields_ = [("shapes", C.c_void_p), ("vels", C.c_void_p), ("index", C.c_void_p), ("count", C.c_int32)]


class fg_final(C.Structure):
    """Terminal block (the ``*_final`` entry points and ``fg_final_obs``): device arrays shaped like the state that
    receive the post-step state of every env whose episode ends in an auto-resetting step."""
    _fields_ = [("pos", C.c_void_p), ("vel", C.c_void_p), ("comm", C.c_void_p), ("ideal_shape", C.c_void_p),
                ("ideal_vel", C.c_void_p), ("landmarks", C.c_void_p)]


class fg_per(C.Structure):
    """Prioritized-replay sum tree (the ``fg_per_*`` entry points): device arrays of caller-owned memory sized by
    ``fg_per_layout``."""
    _fields_ = [("leaf", C.c_void_p), ("sum", C.c_void_p), ("min", C.c_void_p), ("max_leaf", C.c_void_p),
                ("stamp", C.c_void_p), ("prev", C.c_void_p), ("scratch", C.c_void_p),
                ("slots", C.c_longlong), ("envs", C.c_longlong)]


_lib = None


def lib_path():
    return os.environ.get("FG_B200_LIB", _build.LIB_PATH)


def load():
    """Load the shared library (once).  Raises NativeError when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.isfile(path):
        raise NativeError(
            "%s not found: the CUDA extension is not built (run `python -c 'import "
            "__graft_entry__ as g; g.build()'`). There is no CPU fallback." % path)
    lib = C.CDLL(path)
    P, I, U64, U32, VP = C.POINTER, C.c_int, C.c_uint64, C.c_uint32, C.c_void_p
    lib.fg_abi_version.restype = I
    lib.fg_last_error.restype = C.c_char_p
    lib.fg_device_info.argtypes = [P(I), P(I), P(I)]
    lib.fg_launch_geometry.argtypes = [I, P(I), P(I)]
    lib.fg_set_option.argtypes = [C.c_char_p, I]
    lib.fg_get_option.argtypes = [C.c_char_p, P(I)]
    for sfx in ("", "_f64"):
        getattr(lib, "fg_world_step" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, U64, U32, U32, VP]
        getattr(lib, "fg_obs_reward" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, VP]
        getattr(lib, "fg_step_fused" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, I, I, I, U64, U32, U32, VP]
        getattr(lib, "fg_step_policy" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, I, I, I, U64, U32, U32, VP]
        getattr(lib, "fg_reset" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, VP, U64, U32, U32, VP]
        getattr(lib, "fg_step_fused_targets" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, I, I, I, U64, U32, U32, VP, P(fg_targets)]
        getattr(lib, "fg_step_policy_targets" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, I, I, I, U64, U32, U32, VP, P(fg_targets)]
        getattr(lib, "fg_reset_targets" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, VP, U64, U32, U32, VP, P(fg_targets)]
        getattr(lib, "fg_step_fused_final" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, I, I, I, U64, U32, U32, VP, P(fg_targets), P(fg_final)]
        getattr(lib, "fg_step_policy_final" + sfx).argtypes = \
            [P(fg_params), P(fg_buffers), I, I, I, I, I, I, I, U64, U32, U32, VP, P(fg_targets), P(fg_final)]
        getattr(lib, "fg_final_obs" + sfx).argtypes = [P(fg_params), P(fg_final), VP, VP, I, I, I, I, VP]
        getattr(lib, "fg_obs_gather" + sfx).argtypes = \
            [P(fg_params), P(fg_final), C.c_longlong, VP, I, VP, I, I, I, VP]
        getattr(lib, "fg_per_sample" + sfx).argtypes = \
            [P(fg_per), VP, I, C.c_double, VP, VP, VP, I, I, VP, VP, VP, VP, VP, VP, VP, VP, VP, VP]
        getattr(lib, "fg_gae" + sfx).argtypes = [VP, VP, VP, VP, VP, VP, I, C.c_longlong, I, C.c_double, C.c_double, VP]
        getattr(lib, "fg_random_actions" + sfx).argtypes = [VP, I, I, U64, U32, U32, VP, VP]
        getattr(lib, "fg_policy_bfs" + sfx).argtypes = [VP, VP, VP, VP, I, I, I, VP]
        getattr(lib, "fg_pair_distances" + sfx).argtypes = [VP, VP, I, I, VP, VP, VP, VP, VP]
    LL = C.c_longlong
    lib.fg_per_layout.argtypes = [LL, LL, P(LL), P(I), P(LL)]
    lib.fg_per_fill.argtypes = [P(fg_per), LL, LL, LL, I, LL, VP]
    lib.fg_per_update.argtypes = [P(fg_per), VP, VP, VP, I, I, C.c_double, C.c_double, VP]
    lib.fg_obs_to_host.argtypes = [VP, VP, VP, VP, I, I, I, I, I, I, VP]
    lib.fg_fp32_probe.argtypes = [I, I, I, VP, VP]
    lib.fg_write_probe.argtypes = [I, VP, C.c_ulonglong, C.c_uint, I, VP]
    for name in EXPORTS:
        if name != "fg_last_error":
            getattr(lib, name).restype = I
    if lib.fg_abi_version() != FG_ABI_VERSION:
        raise NativeError("ABI mismatch: library %d, binding %d" % (lib.fg_abi_version(), FG_ABI_VERSION))
    _lib = lib
    return lib


def set_option(name, value):
    """A/B switch of the library (include/formation_gym_b200.h fg_set_option); tests and profiling only."""
    check(load().fg_set_option(name.encode(), int(value)), "fg_set_option")


def get_option(name):
    v = C.c_int()
    check(load().fg_get_option(name.encode(), C.byref(v)), "fg_get_option")
    return v.value


class options(object):
    """``with options(force_tile_kernel=1): ...`` -- set A/B switches for a block and restore them after."""

    def __init__(self, **kw):
        self.kw, self.old = kw, {}

    def __enter__(self):
        for k, v in self.kw.items():
            self.old[k] = get_option(k)
            set_option(k, v)
        return self

    def __exit__(self, *exc):
        for k, v in self.old.items():
            set_option(k, v)
        return False


def check(rc, what):
    if rc != 0:
        msg = load().fg_last_error().decode("utf-8", "replace")
        raise NativeError("%s failed (%d): %s" % (what, rc, msg))


def make_params(dt=0.1, damping=0.25, contact_force=1e2, contact_margin=1e-3, sensitivity=5.0,
                agent_size=0.03, mass=1.0, accel=None, max_speed=None, u_noise=None, c_noise=None,
                collide=True, silent=True, world_length=100, walls=(), action_prescaled=False,
                num_obs=0, obs_range=0.0, num_obstacles=0, obstacle_size=0.15, obstacle_mass=1.0,
                obstacle_floor=-2.2, obstacle_fall_vy=-1.0, num_landmarks=0):
    """fg_params from World/Agent attributes (formation_gym/core.py:45-139 defaults)."""
    p = fg_params()
    p.dt, p.damping, p.contact_force, p.contact_margin = dt, damping, contact_force, contact_margin
    p.sensitivity, p.agent_size, p.mass = sensitivity, agent_size, mass
    p.accel = 0.0 if accel is None else float(accel)
    p.has_accel = 0 if accel is None else 1
    p.max_speed = 0.0 if max_speed is None else float(max_speed)
    p.has_max_speed = 0 if max_speed is None else 1
    p.u_noise = float(u_noise) if u_noise else 0.0
    p.c_noise = float(c_noise) if c_noise else 0.0
    p.collide, p.silent, p.world_length = int(bool(collide)), int(bool(silent)), int(world_length)
    p.action_prescaled = int(bool(action_prescaled))
    p.num_obs, p.obs_range = int(num_obs), float(obs_range)
    p.num_obstacles, p.obstacle_size, p.obstacle_mass = int(num_obstacles), float(obstacle_size), float(obstacle_mass)
    p.obstacle_floor, p.obstacle_fall_vy = float(obstacle_floor), float(obstacle_fall_vy)
    p.num_landmarks = int(num_landmarks)
    walls = list(walls)
    if len(walls) > FG_MAX_WALLS:
        raise NativeError("at most %d walls are supported" % FG_MAX_WALLS)
    p.n_walls = len(walls)
    for k, w in enumerate(walls):
        orient, axis_pos, e0, e1, width = w[0], w[1], w[2], w[3], w[4]
        hard = w[5] if len(w) > 5 else True
        p.walls[k].orient = 0 if orient in ('H', 0) else 1
        p.walls[k].hard = int(bool(hard))
        p.walls[k].axis_pos, p.walls[k].end0, p.walls[k].end1, p.walls[k].width = axis_pos, e0, e1, width
    return p


def ptr(t):
    """Raw device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeError("expected a CUDA tensor: the kernels have no CPU path")
    if not t.is_contiguous():
        raise NativeError("expected a contiguous tensor")
    return t.data_ptr()


def device_info():
    sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
    check(load().fg_device_info(C.byref(sm), C.byref(ma), C.byref(mi)), "fg_device_info")
    return sm.value, ma.value, mi.value


def launch_geometry(n):
    epc, thr = C.c_int(), C.c_int()
    check(load().fg_launch_geometry(n, C.byref(epc), C.byref(thr)), "fg_launch_geometry")
    return epc.value, thr.value
