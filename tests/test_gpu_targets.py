"""Target banks of formation_hd_env (include/formation_gym_b200.h fg_targets) on the device: every reset path --
fg_reset, the auto-reset of the warp kernel (STD, generic, with the controller compiled in), of the tile kernel and of
the two-kernel controller path -- gives an env the bank task it is told to take, centred with the kernels' own
arithmetic, and changes nothing else; the tasks drawn for out-of-range indices are reproducible, independent of the
kernel and of sharding, and uniform."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from formation_gym import _native as nat  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402
from formation_gym.vec_env import make_vec_env  # noqa: E402
from formation_gym.envs.formation_hd_env import Scenario  # noqa: E402
from oracle import mpe_oracle as mo  # noqa: E402
from oracle import policy_oracle as po  # noqa: E402

DTYPES = [torch.float32, torch.float64]
DT_IDS = ["f32", "f64"]
NPT = {torch.float32: np.float32, torch.float64: np.float64}


def _bank(K, N, seed, dtype):
    rng = np.random.default_rng(seed)
    return (rng.uniform(-1.5, 1.5, (K, N, 2)).astype(NPT[dtype]), rng.uniform(-1, 1, (K, 2)).astype(NPT[dtype]))


def _centred(raw, t):
    """ideal_shape of a bank entry as the kernels compute it: sequential sums in the env's type, one division by N
    each, one subtraction per item (formation_hd_env.py:93)."""
    N = raw.shape[0]
    sx, sy = t(0), t(0)
    for j in range(N):
        sx, sy = t(sx + raw[j, 0]), t(sy + raw[j, 1])
    return np.stack([raw[:, 0] - t(sx / t(N)), raw[:, 1] - t(sy / t(N))], 1).astype(t)


def _h(x):
    return x.cpu().numpy()


def _want(S, dtype):
    return np.stack([_centred(s, NPT[dtype]) for s in S])


def _check_tasks(env, envs, shapes_c, V, idx):
    """Envs `envs` hold task idx[e]: ideal_shape, ideal_vel and the static part of their observation rows."""
    N = env.N
    got_s, got_v, obs = _h(env.ideal_shape), _h(env.ideal_vel), _h(env.obs)
    k = idx[envs]
    assert np.array_equal(got_s[envs], shapes_c[k])
    assert np.array_equal(got_v[envs], V[k])
    assert np.array_equal(obs[envs][:, :, 4 * N - 2:6 * N - 2], np.repeat(shapes_c[k].reshape(len(envs), 1, 2 * N), N, 1))
    assert np.array_equal(obs[envs][:, :, 6 * N - 2:], np.repeat(V[k][:, None, :], N, 1))


def _drive(env, how, n_steps, n_layer):
    if how == "step":
        for _ in range(n_steps):
            env.step(torch.rand(env.E, env.N, 2, device="cuda", dtype=env.dtype) * 2 - 1)
    elif how == "step_random":
        for _ in range(n_steps):
            env.step_random()
    elif how == "rollout":
        env.rollout_random(n_steps)
    else:
        env.step_bfs(n_layer, n_steps=n_steps)


def _run_paths(N, dtype, how, E=64, n_layer=3, K=5, **env_kw):
    """reset() -> masked reset with a rewritten index -> auto-reset of the other half with another index."""
    S, V = _bank(K, N, N + 100 * K, dtype)
    Sc = _want(S, dtype)
    idx = (np.arange(E) * 7 + 3) % K
    env = BatchedFormationEnv("formation_hd_env", E, N, episode_length=3, dtype=dtype, seed=11,
                              target_shapes=S, target_vels=V, target_index=idx, **env_kw)
    assert env.target_index.dtype == torch.int32 and env.target_index.is_cuda
    env.reset()
    _check_tasks(env, np.arange(E), Sc, V, idx)
    _drive(env, how, 1, n_layer)
    odd, even = np.arange(1, E, 2), np.arange(0, E, 2)
    idx2 = (idx + 1) % K
    env.target_index.copy_(torch.as_tensor(idx2))             # in place: read by the next reset in stream order
    mask = np.zeros(E, bool)
    mask[odd] = True
    before = {k: _h(getattr(env, k)) for k in ("pos", "vel", "ideal_shape", "ideal_vel", "step_count")}
    env.reset(mask)
    _check_tasks(env, odd, Sc, V, idx2)
    for k, v in before.items():                               # envs outside the mask are untouched
        assert np.array_equal(_h(getattr(env, k))[even], v[even]), k
    idx3 = (idx + 2) % K
    env.target_index.copy_(torch.as_tensor(idx3))
    _drive(env, how, 2, n_layer)                              # even envs reach step 3 and are reset in-kernel
    assert np.all(_h(env.step_count)[even] == 0) and np.all(_h(env.step_count)[odd] == 2)
    assert np.all(_h(env.done)[even]) and not np.any(_h(env.done)[odd])
    _check_tasks(env, even, Sc, V, idx3)
    assert np.array_equal(_h(env.ideal_shape)[odd], Sc[idx2[odd]])    # running episodes keep their task
    assert np.array_equal(_h(env.ideal_vel)[odd], V[idx2[odd]])
    return env


WARP_N = [3, 4, 8, 9, 16, 27]


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("how", ["step", "step_random", "rollout"])
@pytest.mark.parametrize("N", WARP_N)
def test_fixed_index_warp(N, how, dtype):
    """k_hd_warp: STD (fp32 single steps with the standard buffers), generic (fp64, fp32 rollouts)."""
    _run_paths(N, dtype, how)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("N", [9, 27])
def test_fixed_index_warp_generic_fp32_switch(N, dtype):
    with nat.options(no_std_kernel=1):
        _run_paths(N, dtype, "step_random")


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("how", ["step", "step_random", "rollout"])
@pytest.mark.parametrize("N,force", [(9, 1), (27, 1), (81, 0)])
def test_fixed_index_tile(N, force, how, dtype):
    """The tile kernel k_step: forced at N = 9 / 27, its own territory at N = 81; also with tracked landmarks, which
    receive the raw bank entry."""
    with nat.options(force_tile_kernel=force):
        env = _run_paths(N, dtype, how, E=40)
        S, _ = _bank(5, N, N + 500, dtype)
        env2 = BatchedFormationEnv("formation_hd_env", 8, N, episode_length=2, dtype=dtype, seed=3, track_landmarks=True,
                                   target_shapes=S, target_index=np.arange(8) % 5)
        raw = S[np.arange(8) % 5].astype(np.float64)
        tol = 1e-5 if dtype == torch.float32 else 1e-12
        env2.reset()                                          # raw entry, re-centred once by reset()'s observation
        lm = mo.hd_landmark_shift(_h(env2.pos).astype(np.float64), raw, times=1)
        assert np.abs(_h(env2.landmarks) - lm).max() <= tol
        env2.step_random()
        env2.step_random()                                    # auto-reset: raw entry, then re-centred by the step
        lm = mo.hd_landmark_shift(_h(env2.pos).astype(np.float64), raw, times=1)
        assert np.abs(_h(env2.landmarks) - lm).max() <= tol
    del env


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("N,n", [(3, 3), (4, 2), (8, 2), (16, 4), (9, 3), (27, 3)])
def test_fixed_index_controller(N, n, dtype):
    """step_bfs: one launch per step for (3,3), (4,2), (8,2), (16,4); the step and controller kernels for 9, 27."""
    env = _run_paths(N, dtype, "bfs", n_layer=n)
    want = po.bfs_actions_batch(_h(env.pos).astype(np.float64), _h(env.ideal_shape).astype(np.float64),
                                _h(env.ideal_vel).astype(np.float64), n)
    err = np.abs(_h(env.actions).astype(np.float64) - want).max(axis=(1, 2))
    if dtype == torch.float64:
        assert err.max() <= 1e-11
    else:
        assert (err > 1e-5).mean() <= 0.05                   # samples on a decision boundary may branch differently


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_fixed_index_many_spans(dtype):
    """More spans of 3 envs than the 3 552 resident warps at N = 9: every warp walks several spans."""
    E, N, K = 12000, 9, 6
    S, V = _bank(K, N, 5, dtype)
    Sc = _want(S, dtype)
    idx = np.arange(E) % K
    env = BatchedFormationEnv("formation_hd_env", E, N, episode_length=2, dtype=dtype, seed=2,
                              target_shapes=S, target_vels=V, target_index=idx)
    env.reset()
    _check_tasks(env, np.arange(E), Sc, V, idx)
    idx2 = (idx + 1) % K
    env.target_index.copy_(torch.as_tensor(idx2))
    env.step_random()
    env.step_random()
    assert np.all(_h(env.step_count) == 0)
    _check_tasks(env, np.arange(E), Sc, V, idx2)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("force", [0, 1], ids=["warp", "tile"])
def test_bank_changes_nothing_else(force, dtype):
    """Same seed and ticks: positions, velocities and step counters are bit-identical to a run without a bank; so is
    ideal_vel when the bank has no velocities."""
    E, N = 50, 9
    S, V = _bank(4, N, 9, dtype)
    with nat.options(force_tile_kernel=force):
        for vels in (None, V):
            plain = BatchedFormationEnv("formation_hd_env", E, N, episode_length=3, dtype=dtype, seed=4)
            bank = BatchedFormationEnv("formation_hd_env", E, N, episode_length=3, dtype=dtype, seed=4,
                                       target_shapes=S, target_vels=vels)
            plain.reset()
            bank.reset()
            for t in range(8):
                for k in ("pos", "vel", "step_count"):
                    assert torch.equal(getattr(plain, k), getattr(bank, k)), (t, k)
                if vels is None:
                    assert torch.equal(plain.ideal_vel, bank.ideal_vel)
                else:
                    assert not torch.equal(plain.ideal_vel, bank.ideal_vel)
                plain.step_random()
                bank.step_random()


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("layer", [1, 2])
def test_hierarchical_shapes_observation_reward_and_controller(layer, dtype):
    """The reference's hierarchical targets (Scenario.generate_shape(1): 9 agents, (2): 27): after an in-kernel
    auto-reset the observation rows carry the new task, and observation, reward and the controller's actions match
    the numpy oracles on the read-back state."""
    tol = 1e-5 if dtype == torch.float32 else 1e-9
    g = Scenario().generate_shape(layer).reshape(-1, 2)
    N = g.shape[0]
    S = np.stack([g, -g[:, ::-1]]).astype(NPT[dtype])          # the shape and a mirrored copy
    E = 30
    idx = np.arange(E) % 2
    env = BatchedFormationEnv("formation_hd_env", E, N, episode_length=2, dtype=dtype, seed=8,
                              target_shapes=S, target_index=idx)
    env.reset()
    env.step_random()
    env.target_index.copy_(torch.as_tensor(1 - idx))
    obs, _, done, _ = env.step_random()                        # auto-reset of every env
    assert bool(done.all())
    st = {k: _h(getattr(env, k)).astype(np.float64) for k in ("pos", "vel", "ideal_shape", "ideal_vel")}
    assert np.array_equal(_h(env.ideal_shape), _want(S, dtype)[1 - idx])
    assert np.abs(_h(obs) - mo.hd_observation(st["pos"], st["vel"], st["ideal_shape"], st["ideal_vel"])).max() <= tol
    # one more step from the reset state on recorded actions: obs / reward of the new task
    act = torch.rand(E, N, 2, device="cuda", dtype=dtype) * 2 - 1
    out = mo.hd_env_step(st["pos"], st["vel"], _h(act).astype(np.float64), st["ideal_shape"], st["ideal_vel"],
                         _h(env.step_count), prm=mo.HD_PARAMS)
    obs, rew, _, info = env.step(act)
    assert np.abs(_h(obs) - out["obs"]).max() <= tol
    assert np.abs(_h(info["individual_reward"]) - out["indiv"]).max() <= tol * (10 if layer == 2 else 1)
    R = out["reward"]
    rtol = 1e-6 if dtype == torch.float32 else 1e-13
    assert np.all(np.abs(_h(rew)[:, :, 0] - R[:, None]) <= tol + rtol * np.abs(R[:, None]))
    # the controller on the bank shape
    env.reset()
    act = _h(env.bfs_actions(3)).astype(np.float64)
    want = po.bfs_actions_batch(_h(env.pos).astype(np.float64), _h(env.ideal_shape).astype(np.float64),
                                _h(env.ideal_vel).astype(np.float64), 3)
    err = np.abs(act - want).max(axis=(1, 2))
    if dtype == torch.float64:
        assert err.max() <= 1e-11
    else:
        assert (err > 1e-5).mean() <= 0.05


def _drawn(env):
    """Task of every env, read from a bank whose velocities are (k, 0)."""
    return _h(env.ideal_vel)[:, 0].astype(np.int64)


def _vel_bank(K, N):
    S, _ = _bank(K, N, K, torch.float32)
    return S, np.stack([np.arange(K), np.zeros(K)], 1).astype(np.float32)


def test_draws_are_reproducible_and_kernel_independent():
    E, N, K = 300, 9, 7
    S, V = _vel_bank(K, N)
    runs = []
    for force in (0, 0, 1):
        with nat.options(force_tile_kernel=force):
            env = BatchedFormationEnv("formation_hd_env", E, N, episode_length=2, seed=21, target_shapes=S, target_vels=V)
            env.reset()
            seq = [_drawn(env)]
            for _ in range(2):
                env.step_random()
                env.step_random()
                seq.append(_drawn(env))
            runs.append((np.stack(seq), _h(env.ideal_shape)))
    for r in runs[1:]:
        assert np.array_equal(r[0], runs[0][0]) and np.array_equal(r[1], runs[0][1])
    assert not np.array_equal(runs[0][0][0], runs[0][0][1])  # a new draw at every reset


def test_draws_do_not_depend_on_sharding():
    E, N, K = 200, 4, 7
    S, V = _vel_bank(K, N)

    def run(n, off):
        env = BatchedFormationEnv("formation_hd_env", n, N, episode_length=2, seed=5, env_offset=off,
                                  target_shapes=S, target_vels=V)
        env.reset()
        a = _drawn(env)
        env.step_random()
        env.step_random()
        return np.concatenate([a, _drawn(env)])

    whole = run(E, 0)
    half = [run(E // 2, 0), run(E // 2, E // 2)]
    assert np.array_equal(whole[:E], np.concatenate([half[0][:E // 2], half[1][:E // 2]]))
    assert np.array_equal(whole[E:], np.concatenate([half[0][E // 2:], half[1][E // 2:]]))


def test_draws_are_uniform():
    from scipy.stats import chisquare
    E, N, K = 65536, 3, 7
    S, V = _vel_bank(K, N)
    env = BatchedFormationEnv("formation_hd_env", E, N, episode_length=1, seed=13, target_shapes=S, target_vels=V)
    env.reset()
    at_reset = _drawn(env)
    env.step_random()                                                      # episode length 1: every env auto-resets
    for draws in (at_reset, _drawn(env)):
        counts = np.bincount(draws, minlength=K)
        assert counts.sum() == E and len(counts) == K
        assert chisquare(counts).pvalue > 1e-4, counts


def test_out_of_range_index_means_draw():
    E, N, K = 64, 9, 7
    S, V = _vel_bank(K, N)
    idx = np.array([-1, K, 2 * K, -7, 3] * 12 + [0, 1, 2, 6])
    free = BatchedFormationEnv("formation_hd_env", E, N, episode_length=2, seed=6, target_shapes=S, target_vels=V)
    some = BatchedFormationEnv("formation_hd_env", E, N, episode_length=2, seed=6, target_shapes=S, target_vels=V,
                               target_index=idx)
    for _ in range(2):
        free.reset()
        some.reset()
        ok = (idx >= 0) & (idx < K)
        assert np.array_equal(_drawn(some)[~ok], _drawn(free)[~ok])
        assert np.array_equal(_drawn(some)[ok], idx[ok])
        free.step_random(); free.step_random()                             # noqa: E702
        some.step_random(); some.step_random()                             # noqa: E702
        assert np.array_equal(_drawn(some)[~ok], _drawn(free)[~ok])
        assert np.array_equal(_drawn(some)[ok], idx[ok])


def test_vec_env_host_obs_stays_identical_across_auto_resets():
    E, N, K = 64, 9, 3
    S, V = _bank(K, N, 1, torch.float32)
    venv = make_vec_env("formation_hd_env", E, N, episode_length=3, target_shapes=S, target_vels=V,
                        target_index=np.arange(E) % K)
    venv.reset()
    rng = np.random.default_rng(0)
    seen = set()
    for t in range(10):
        if t == 4:
            venv.env.target_index.copy_(torch.as_tensor((np.arange(E) + 1) % K))   # curriculum step between steps
        obs, _, done, _ = venv.step(rng.uniform(-1, 1, (E, N, 2)).astype(np.float32))
        assert np.array_equal(obs, _h(venv.env.obs))
        seen.add(obs[0, 0, 4 * N - 2:6 * N - 2].tobytes())
    assert len(seen) == 2                                                  # the curriculum reached the host rows


def test_graph_replays_read_the_index_in_stream_order():
    E, N, K = 32, 3, 4
    S, V = _bank(K, N, 2, torch.float32)
    env = BatchedFormationEnv("formation_hd_env", E, N, episode_length=2, seed=1, target_shapes=S, target_vels=V,
                              target_index=np.zeros(E, np.int32))
    env.reset()
    g = env.capture_steps(2, fused_random=True)                            # both steps end at an episode end
    for k in (1, 3, 2):
        env.target_index.fill_(k)
        g.replay()
        assert np.array_equal(_h(env.ideal_vel), np.repeat(V[k][None], E, 0))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_state_dict_carries_the_index(dtype):
    E, N = 10, 4
    S, V = _bank(3, N, 4, dtype)
    env = BatchedFormationEnv("formation_hd_env", E, N, dtype=dtype, target_shapes=S, target_index=np.arange(E) % 3)
    env.reset()
    sd = env.state_dict()
    assert torch.equal(sd["target_index"], torch.as_tensor(np.arange(E) % 3, dtype=torch.int32, device="cuda"))
    env.target_index.fill_(-1)
    env.load_state_dict(sd)
    assert torch.equal(env.target_index, sd["target_index"])
    plain = BatchedFormationEnv("formation_hd_env", E, N, dtype=dtype)
    assert "target_index" not in plain.state_dict() and plain.target_index is None
