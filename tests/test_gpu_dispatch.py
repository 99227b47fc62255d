"""Which kernel instantiation each entry point launches, read from torch.profiler around one call.

The host layer picks among the warp-autonomous kernels (k_hd_warp, k_lm_warp), the tile kernels (k_step,
k_step_obst) and their STD / EXT / POL instantiations from the scenario, N, dtype, the buffers and the A/B switches.
These rows pin that choice, so a change to the host code cannot move a configuration to another kernel unnoticed."""
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

from formation_gym import _native as nat  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402

HD, PARTIAL, RANGE, OBST, BASIC = ("formation_hd_env", "formation_hd_partial_env", "formation_hd_partial_range_env",
                                   "formation_hd_obs_env", "basic_formation_env")
_KERNEL = re.compile(r"\b(k_\w+)<([^<>]*)>")


def _launched(fn):
    """(kernel, template arguments) of every kernel fn() launches, in launch order.  fn runs once before the profiled
    call, so one-time work (step_bfs's first controller launch) stays out of the list."""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = []
    for e in sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                    key=lambda e: e.time_range.start):
        m = _KERNEL.search(e.name)
        if m:
            out.append((m.group(1), tuple(a.strip() for a in m.group(2).split(","))))
    return out


def _k(name, *args):
    return (name, tuple(str(a).lower() if isinstance(a, bool) else str(a) for a in args))


def _env(scen, N, dtype=torch.float32, **kw):
    env = BatchedFormationEnv(scen, 1024, N, dtype=dtype, seed=1, **kw)
    env.reset()
    return env


# k_hd_warp<T, N, WOBS, SCN, STD, POL, EXT>; k_lm_warp<T, N, L, SCN, NOBS, STD, EXT>;
# k_step<T, SCN, PHYS, OBSREW, HET, OM, FP, EXT>; k_step_obst<T, PHYS, OBSREW, EXT>
@pytest.mark.parametrize("N", [3, 9, 27, 32])
def test_hd_warp_std(N):
    env = _env(HD, N)
    assert _launched(env.step_random) == [_k("k_hd_warp", "float", N, True, 0, True, 0, False)]
    with nat.options(no_std_kernel=1):
        assert _launched(env.step_random) == [_k("k_hd_warp", "float", N, True, 0, False, 0, False)]
    env64 = _env(HD, N, torch.float64)
    assert _launched(env64.step_random) == [_k("k_hd_warp", "double", N, True, 0, False, 0, False)]


@pytest.mark.parametrize("N,om,fp", [(10, 2, False), (81, 2, True), (243, 2, True)])
def test_hd_tile(N, om, fp):
    env = _env(HD, N)
    assert _launched(env.step_random) == [_k("k_step", "float", 0, True, True, False, om, fp, False)]


def test_basic():
    assert _launched(_env(BASIC, 3).step_random) == [_k("k_hd_warp", "float", 3, True, 1, True, 0, False)]
    assert _launched(_env(BASIC, 4).step_random) == [_k("k_step", "float", 1, True, True, False, 3, False, False)]


@pytest.mark.parametrize("scen,N,expect", [
    (PARTIAL, 4, _k("k_lm_warp", "float", 4, 5, 2, 3, True, False)),
    (RANGE, 5, _k("k_lm_warp", "float", 5, 4, 3, 0, True, False)),
    (OBST, 4, _k("k_lm_warp", "float", 4, 7, 4, 3, True, False)),
    (OBST, 10, _k("k_step_obst", "float", True, True, False)),
])
def test_landmark_scenarios(scen, N, expect):
    assert _launched(_env(scen, N).step_random) == [expect]


@pytest.mark.parametrize("scen,N,expect", [
    (HD, 9, _k("k_hd_warp", "float", 9, True, 0, True, 0, True)),
    (HD, 10, _k("k_step", "float", 0, True, True, False, 2, False, True)),
    (PARTIAL, 4, _k("k_lm_warp", "float", 4, 5, 2, 3, True, True)),
    (OBST, 10, _k("k_step_obst", "float", True, True, True)),
])
def test_record_final_ext(scen, N, expect):
    assert _launched(_env(scen, N, record_final=True).step_random) == [expect]


def test_step_bfs():
    env = _env(HD, 3)
    assert _launched(env.step_bfs) == [_k("k_hd_warp", "float", 3, True, 0, True, 3, False)]
    env = _env(HD, 9)
    assert _launched(env.step_bfs) == [_k("k_hd_warp", "float", 9, True, 0, True, 0, False),
                                       _k("k_policy_bfs", "float", 3, 2)]


def test_observation_passes():
    obs_pass = _k("k_step", "float", 0, False, True, False, 3, False, False)
    env = _env(HD, 9, record_final=True)
    assert _launched(env.observe) == [obs_pass]
    env.step_random()
    assert _launched(env.final_observation) == [_k("k_step", "float", 0, False, True, False, 3, False, True)]
    states = {k: getattr(env, k).clone() for k in env.state_record_keys()}
    rows = torch.arange(0, 1024, 3, device="cuda", dtype=torch.int64)
    assert _launched(lambda: env.gather_observations(states, rows)) == [
        _k("k_step", "float", 0, False, True, False, 3, False, True)]
    env = _env(OBST, 4, record_final=True)
    assert _launched(env.observe) == [_k("k_step_obst", "float", False, True, False)]
    env.step_random()
    assert _launched(env.final_observation) == [_k("k_step_obst", "float", False, True, True)]


def test_reset():
    assert _launched(_env(HD, 9).reset) == [_k("k_reset", "float", 0),
                                            _k("k_step", "float", 0, False, True, False, 3, False, False)]
    assert _launched(_env(OBST, 4).reset) == [_k("k_reset_obst", "float"),
                                              _k("k_step_obst", "float", False, True, False)]


def test_force_tile_kernel():
    env = _env(HD, 9)
    with nat.options(force_tile_kernel=1):
        assert _launched(env.step_random) == [_k("k_step", "float", 0, True, True, False, 3, False, False)]
