"""Terminal blocks (include/formation_gym_b200.h fg_final) on the device: every step kernel family copies the post-step
state of an env whose episode ends into the block before its auto-reset overwrites it, bit-identical to a run without
auto-reset; fg_final_obs turns the block into the observation rows that run returns; and nothing else a step computes
changes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from formation_gym import _native as nat  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402
from formation_gym.vec_env import make_vec_env  # noqa: E402
from oracle import mpe_oracle as mo  # noqa: E402

DTYPES = [torch.float32, torch.float64]
DT_IDS = ["f32", "f64"]
EP = 4                                                     # episode length of most cases
STATE = ("pos", "vel", "comm", "ideal_shape", "ideal_vel", "landmarks")
OUTPUTS = ("pos", "vel", "comm", "obs", "reward", "indiv", "done", "step_count", "ep_return", "ep_collisions",
           "stats", "nan_flag", "ideal_shape", "ideal_vel", "landmarks", "landmark_vel", "actions")


def _h(x):
    return x.cpu().numpy()


def _bank(N, dtype, E):
    rng = np.random.default_rng(5)
    return dict(target_shapes=rng.uniform(-1.5, 1.5, (3, N, 2)), target_vels=rng.uniform(-1, 1, (3, 2)),
                target_index=np.arange(E) % 4 - 1)         # -1: drawn, else a task


def _make(scn, E, N, dtype, auto_reset, record_final=False, bank=False, episode_length=EP, **kw):
    if bank:
        kw.update(_bank(N, dtype, E))
    env = BatchedFormationEnv(scn, E, N, episode_length, dtype=dtype, seed=21, auto_reset=auto_reset,
                              record_final=record_final, **kw)
    env.reset()
    env.pos.mul_(0.3)                                      # dense: contacts and reward collisions occur
    env.observe()
    return env


def _advance(env, how, n_layer=3, s=0):
    """One step; two envs advanced alike draw the same actions (same seed and tick, or the same generator seed)."""
    if how == "step":
        if env.silent:
            env.sample_actions()
        else:
            env.actions.uniform_(-1, 1, generator=torch.Generator(device=env.device).manual_seed(s))
        return env.step(env.actions)
    if how == "random":
        return env.step_random(record_actions=True)
    return env.step_bfs(n_layer)


def _check_block(A, B, ended):
    """A's terminal block and terminal observation rows of the envs `ended` equal B's state and rows."""
    torch.cuda.synchronize()
    for k in STATE:
        blk = getattr(A, "final_" + k)
        if blk is None:
            continue
        want = getattr(B, k)
        assert np.array_equal(_h(blk)[ended], _h(want)[ended], equal_nan=True), k
    fo = A.final_observation()
    if B.obs is not None:
        assert np.array_equal(_h(fo)[ended], _h(B.obs)[ended], equal_nan=True), "final_observation"
    return fo


def _terminal_pair(scn, E, N, dtype, how="step", bank=False, opts=None, n_layer=3, **kw):
    """Run A (record_final, auto-reset) and B (no auto-reset) with the same seed and actions through one episode and
    compare A's terminal block at the terminal step with B's state."""
    with nat.options(**(opts or {})):
        A = _make(scn, E, N, dtype, True, record_final=True, bank=bank, **kw)
        B = _make(scn, E, N, dtype, False, bank=bank, **kw)
        for s in range(EP):
            _advance(A, how, n_layer, s)
            _advance(B, how, n_layer, s)
        torch.cuda.synchronize()
        done = _h(A.done)[:, 0]
        assert done.all() and np.array_equal(_h(B.done)[:, 0], done)
        _check_block(A, B, np.arange(E))
        # A went on with the reset state: not B's
        assert not np.array_equal(_h(A.pos), _h(B.pos))


# ------------------------------------------------------------------ 1. bit-exact against a run without auto-reset
HD_CASES = [(3, 1001), (9, 1000), (9, 257), (27, 65), (27, 1)]


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("N,E", HD_CASES)
@pytest.mark.parametrize("std", [1, 0], ids=["std", "generic"])
@pytest.mark.parametrize("how", ["step", "random"])
def test_warp_hd_terminal_block(N, E, dtype, std, how):
    _terminal_pair("formation_hd_env", E, N, dtype, how, opts=dict(no_std_kernel=1 - std))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("N,E", [(9, 1000), (3, 77)])
def test_warp_hd_terminal_block_with_bank(N, E, dtype):
    _terminal_pair("formation_hd_env", E, N, dtype, "random", bank=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("how", ["step", "random"])
def test_warp_basic_terminal_block(dtype, how):
    _terminal_pair("basic_formation_env", 1003, 3, dtype, how)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("N,E,kw", [(9, 300, {}), (27, 40, {}), (64, 9, {}), (100, 5, {}), (9, 70, dict(silent=False)),
                                    (9, 50, dict(track_landmarks=True))],
                         ids=["n9", "n27", "n64", "n100", "comm", "lm"])
@pytest.mark.parametrize("bank", [False, True], ids=["plain", "bank"])
def test_tile_hd_terminal_block(N, E, kw, dtype, bank):
    """The tile kernel: scalar pair loops, packed pairs with cell lists (N >= 64, fp32), non-silent agents, tracked
    landmarks, with and without a bank."""
    how = "step" if kw.get("silent", True) is False else "random"
    _terminal_pair("formation_hd_env", E, N, dtype, how, bank=bank, opts=dict(force_tile_kernel=1), **kw)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N", [("basic_formation_env", 5), ("formation_hd_partial_env", 6),
                                   ("formation_hd_partial_range_env", 5), ("formation_hd_obs_env", 4)])
def test_tile_landmark_scenarios_terminal_block(scn, N, dtype):
    _terminal_pair(scn, 301, N, dtype, "random", opts=dict(force_tile_kernel=1))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N,E", [("formation_hd_partial_env", 4, 1001), ("formation_hd_partial_env", 9, 33),
                                     ("formation_hd_partial_range_env", 4, 1001), ("formation_hd_obs_env", 4, 1001),
                                     ("formation_hd_obs_env", 7, 19)])
@pytest.mark.parametrize("how", ["step", "random"])
def test_lm_warp_terminal_block(scn, N, E, dtype, how):
    _terminal_pair(scn, E, N, dtype, how)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_obstacle_tile_terminal_block(dtype):
    """k_step_obst at N > 9 (no warp instantiation)."""
    _terminal_pair("formation_hd_obs_env", 150, 12, dtype, "random")


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("N,n,E", [(3, 3, 1001), (4, 2, 300), (9, 3, 300), (16, 4, 65)],
                         ids=["fused3", "fused4", "two_kernel9", "fused16"])
@pytest.mark.parametrize("bank", [False, True], ids=["plain", "bank"])
def test_step_bfs_terminal_block(N, n, E, dtype, bank):
    """The controller-fused warp kernel and the two-kernel controller path (N = 9)."""
    _terminal_pair("formation_hd_env", E, N, dtype, "bfs", bank=bank, n_layer=n)


def test_more_spans_than_resident_warps():
    """A persistent warp walks several spans: N = 3, 150001 envs (ragged last span)."""
    _terminal_pair("formation_hd_env", 150001, 3, torch.float32, "random")
    _terminal_pair("basic_formation_env", 150001, 3, torch.float32, "random")


# ------------------------------------------------------------------ 2. no side effects
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N,opts", [("formation_hd_env", 9, {}), ("formation_hd_env", 9, dict(force_tile_kernel=1)),
                                        ("basic_formation_env", 3, {}), ("formation_hd_partial_env", 4, {}),
                                        ("formation_hd_obs_env", 4, {}), ("formation_hd_obs_env", 4,
                                                                          dict(force_tile_kernel=1))],
                         ids=["hd_warp", "hd_tile", "basic", "partial", "obs_env", "obs_tile"])
def test_block_changes_nothing_else(scn, N, opts, dtype):
    """Several episodes, step and step_random, with and without a block (final_observation called every step):
    every regular output, the state, the statistics and nan_flag stay bit for bit the same."""
    E = 515
    with nat.options(**opts):
        A = _make(scn, E, N, dtype, True, record_final=True)
        C_ = _make(scn, E, N, dtype, True)
        for s in range(3 * EP + 1):
            how = "step" if s % 2 else "random"
            _advance(A, how)
            A.final_observation()
            _advance(C_, how)
            torch.cuda.synchronize()
            for k in OUTPUTS:
                a, c = getattr(A, k), getattr(C_, k)
                if a is None:
                    assert c is None
                    continue
                if k == "stats":                           # (per-warp partial sums meet in global atomics: any order)
                    assert torch.equal(a[[0, 3]], c[[0, 3]]), s
                    assert torch.allclose(a, c, rtol=1e-12, atol=0), s
                    continue
                assert torch.equal(a, c), (s, k)
        assert A.episode_stats()["episodes"] == 3 * E


# ------------------------------------------------------------------ 3. staggered episodes
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N,opts", [("formation_hd_env", 9, {}), ("formation_hd_env", 9, dict(force_tile_kernel=1)),
                                        ("formation_hd_partial_range_env", 4, {}), ("formation_hd_obs_env", 4, {})],
                         ids=["hd_warp", "hd_tile", "range", "obs_env"])
def test_staggered_episodes(scn, N, opts, dtype):
    """After reset(mask) on half of the envs only the envs that end get block entries; the others keep a sentinel."""
    E = 640
    with nat.options(**opts):
        A = _make(scn, E, N, dtype, True, record_final=True)
        B = _make(scn, E, N, dtype, False)
        for s in range(2):
            A.step_random(record_actions=True)
            B.step(A.actions)
        mask = torch.zeros(E, dtype=torch.bool, device=A.device)
        mask[::2] = True
        A.reset(mask)
        B.reset(mask)                                      # same seed and tick: same reset state
        for k in STATE:
            if getattr(A, "final_" + k) is not None:
                getattr(A, "final_" + k).fill_(1234.5)
        for s in range(EP - 2):
            A.step_random(record_actions=True)
            B.step(A.actions)
        torch.cuda.synchronize()
        ended = _h(A.done)[:, 0]
        assert np.array_equal(ended, ~_h(mask)) and np.array_equal(_h(B.done)[:, 0], ended)
        idx = np.nonzero(ended)[0]
        fo = _check_block(A, B, idx)
        for k in STATE:
            blk = getattr(A, "final_" + k)
            if blk is not None:
                assert (_h(blk)[~ended] == 1234.5).all(), k
        # the mask rows only: a second call after a step that ended nothing writes nothing
        before = fo.clone()
        A.step_random()
        A.final_observation()
        torch.cuda.synchronize()
        assert not _h(A.done)[:, 0].any()
        assert torch.equal(A.final_observation(), before)


# ------------------------------------------------------------------ 4. reference tie-in
def test_terminal_observation_matches_the_oracle():
    """hd N = 9, fp64: the terminal observation after world_length steps is the reference's observation of the state
    it steps to from the same state (traj25 bar 1e-9)."""
    E, N = 64, 9
    A = _make("formation_hd_env", E, N, torch.float64, True, record_final=True)
    for s in range(EP - 1):
        A.step_random()
    torch.cuda.synchronize()
    st = {k: _h(getattr(A, k)).copy() for k in ("pos", "vel", "ideal_shape", "ideal_vel")}
    A.step_random(record_actions=True)
    ref = mo.hd_env_step(st["pos"], st["vel"], _h(A.actions), st["ideal_shape"], st["ideal_vel"], np.zeros(E))
    fo = _h(A.final_observation())
    assert _h(A.done).all()
    assert np.abs(fo - ref["obs"]).max() <= 1e-9
    assert np.abs(_h(A.final_pos) - ref["pos"]).max() <= 1e-9


# ------------------------------------------------------------------ 5. CUDA graphs and CudaVecEnv
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_graph_replay_matches_host_launches(dtype):
    E, N = 2000, 9
    H = _make("formation_hd_env", E, N, dtype, True, record_final=True)
    G = _make("formation_hd_env", E, N, dtype, True, record_final=True)
    H.use_device_tick(True)
    seen = []

    def policy(env):
        seen.append(env.final_observation())
        env.sample_actions()

    graph = G.capture_steps(1, policy=policy)
    fo_g = G._final_obs
    # the capture's warm-up ran one step already: the host-launched twin does the same
    H.final_observation()
    H.sample_actions()
    H.step(H.actions)
    for s in range(3 * EP - 1):                            # 3 * EP steps in all
        graph.replay()
        H.final_observation()
        H.sample_actions()
        H.step(H.actions)
        torch.cuda.synchronize()
        for k in ("pos", "vel", "obs", "reward", "done"):
            assert torch.equal(getattr(G, k), getattr(H, k)), (s, k)
        for k in ("pos", "vel", "ideal_shape", "ideal_vel"):
            assert torch.equal(getattr(G, "final_" + k), getattr(H, "final_" + k)), (s, k)
    ended = _h(H.done)[:, 0]
    assert ended.all()                                     # the last step ends the third episodes
    G.final_observation(); H.final_observation()
    torch.cuda.synchronize()
    assert seen[0] is fo_g
    assert torch.equal(G._final_obs, H._final_obs)


@pytest.mark.parametrize("to_numpy", [True, False], ids=["numpy", "torch"])
@pytest.mark.parametrize("scn,N", [("formation_hd_env", 9), ("formation_hd_partial_env", 4)])
def test_vec_env_terminal_observation(scn, N, to_numpy):
    E = 100
    V = make_vec_env(scn, E, N, EP, to_numpy=to_numpy, seed=4, record_final=True)
    W = make_vec_env(scn, E, N, EP, to_numpy=to_numpy, seed=4)
    B = BatchedFormationEnv(scn, E, N, EP, seed=4, auto_reset=False)
    V.reset(); W.reset(); B.reset()
    for s in range(2 * EP):
        act = V.sample_actions()
        act = act.copy() if to_numpy else act.clone()
        o1, r1, d1, i1 = V.step(act)
        o2, r2, d2, i2 = W.step(act)
        B.step(torch.as_tensor(act, device=B.device))
        conv = (lambda x: np.asarray(x)) if to_numpy else _h
        assert np.array_equal(conv(o1), conv(o2)) and np.array_equal(conv(r1), conv(r2))
        assert i2.terminal_observation is None and set(i2[0][0]) == {"individual_reward"}
        assert i1[0][0]["individual_reward"] == i2[0][0]["individual_reward"]
        if (s + 1) % EP:
            assert i1.terminal_observation is None and set(i1[3][1]) == {"individual_reward"}
            continue
        assert conv(d1)[:, 0].all()
        tobs = conv(i1.terminal_observation)
        assert np.array_equal(tobs, _h(B.obs))
        row = i1[3][1]["terminal_observation"]
        assert np.array_equal(conv(row), _h(B.obs)[3, 1])
        if to_numpy:
            assert isinstance(i1.terminal_observation, np.ndarray)
        B.load_state_dict(V.env.state_dict())              # B follows V's auto-reset


# ------------------------------------------------------------------ 6. NaN envs
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("opts", [{}, dict(force_tile_kernel=1)], ids=["warp", "tile"])
def test_nan_env_terminal_state_copied_as_is(opts, dtype):
    """Coincident agents make the contact force NaN (core.py:312); the NaN terminal state is copied as it is."""
    E, N = 40, 9
    with nat.options(**opts):
        A = _make("formation_hd_env", E, N, dtype, True, record_final=True)
        B = _make("formation_hd_env", E, N, dtype, False)
        for env in (A, B):
            env.pos[7, 1] = env.pos[7, 0]
            env.pos[E - 1, 4] = env.pos[E - 1, 2]
        for s in range(EP):
            A.step_random(record_actions=True)
            B.step(A.actions)
        torch.cuda.synchronize()
        assert _h(A.nan_flag)[[7, E - 1]].all() and torch.equal(A.nan_flag, B.nan_flag)
        assert np.isnan(_h(A.final_pos)[7]).any()
        _check_block(A, B, np.arange(E))
        assert np.isfinite(_h(A.pos)).all()                 # the reset state is finite again
