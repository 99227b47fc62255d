"""State-record replay on the device: fg_obs_gather turns sampled state records into the observation rows the steps
returned, bit for bit, for every kernel family; out-of-range indices give NaN rows; records past 2^32 bytes are
addressed correctly; StateReplayBuffer builds (s, a, r, s', done) transitions with the right chains, terminal states
and wrap-around; and a buffer changes nothing the env computes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from formation_gym import StateReplayBuffer  # noqa: E402
from formation_gym import _native as nat  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402

DTYPES = [torch.float32, torch.float64]
DT_IDS = ["f32", "f64"]
EP = 4


def _h(x):
    return x.cpu().numpy()


def _make(scn, E, N, dtype, bank=False, **kw):
    if bank:
        rng = np.random.default_rng(5)
        kw.update(target_shapes=rng.uniform(-1.5, 1.5, (3, N, 2)), target_vels=rng.uniform(-1, 1, (3, 2)),
                  target_index=np.arange(E) % 4 - 1)
    env = BatchedFormationEnv(scn, E, N, EP, dtype=dtype, seed=21, auto_reset=True, record_final=True, **kw)
    env.reset()
    env.pos.mul_(0.3)                                      # dense: contacts and reward collisions occur
    env.observe()
    return env


def _step(env, how, s, n_layer=3):
    """One step; returns the actions it ran on."""
    if how == "step":
        if env.silent:
            env.sample_actions()
        else:
            env.actions.uniform_(-1, 1, generator=torch.Generator(device=env.device).manual_seed(s))
        env.step(env.actions)
        return env.actions
    if how == "random":
        env.step_random(record_actions=True)
        return env.actions
    act = env.actions.clone() if env._bfs_primed == n_layer else env.bfs_actions(n_layer).clone()
    env.step_bfs(n_layer)                                  # (env.actions now holds the NEXT actions)
    return act


def _record(env, steps, how="random", capacity=None, n_layer=3):
    """A buffer over `steps` auto-resetting steps, and the observation every record of it must decode to: S records
    the obs the step returned (the reset obs for the chain start), F records the terminal observation (ended envs)."""
    buf = StateReplayBuffer(env, capacity or steps + 1)
    T, E = buf.capacity, env.E
    want = torch.full((buf.num_records, env.N, env.D), float("nan"), dtype=env.dtype, device=env.device)
    ended = torch.zeros(buf.num_records, dtype=torch.bool, device=env.device)
    buf.mark_start()
    want[0:E] = env.obs
    for s in range(steps):
        j = buf._next
        buf.add(_step(env, how, s, n_layer))
        want[j * E:(j + 1) * E] = env.obs
        want[(T + j) * E:(T + j + 1) * E] = env.final_observation()
        ended[(T + j) * E:(T + j + 1) * E] = env.done[:, 0]
    S = torch.arange(T * E, device=env.device)
    return buf, want, torch.cat([S, torch.nonzero(ended).flatten()])


def _check_decode(env, buf, want, valid, B=6000, seed=3):
    g = torch.Generator(device=env.device).manual_seed(seed)
    rows = valid[torch.randint(0, valid.shape[0], (B,), device=env.device, generator=g)]   # repeats, any order
    got = env.gather_observations(buf.states, rows)
    torch.cuda.synchronize()
    assert torch.equal(got, want[rows])
    # every record at least once, in reverse order
    got = env.gather_observations(buf.states, valid.flip(0))
    assert torch.equal(got, want[valid.flip(0)])


# ------------------------------------------------------------------ 1. bit-exact decode, every kernel family
CASES = {
    "hd3_std": ("formation_hd_env", 3, 1001, {}, {}), "hd3_generic": ("formation_hd_env", 3, 1001, {}, dict(no_std_kernel=1)),
    "hd9_std": ("formation_hd_env", 9, 1000, {}, {}), "hd9_generic": ("formation_hd_env", 9, 1000, {}, dict(no_std_kernel=1)),
    "hd27_std": ("formation_hd_env", 27, 65, {}, {}), "hd27_generic": ("formation_hd_env", 27, 65, {}, dict(no_std_kernel=1)),
    "basic3": ("basic_formation_env", 3, 1003, {}, {}),
    "partial4": ("formation_hd_partial_env", 4, 1001, {}, {}),
    "range4": ("formation_hd_partial_range_env", 4, 1001, {}, {}),
    "obs_env4": ("formation_hd_obs_env", 4, 1001, {}, {}),
    "obs_env12": ("formation_hd_obs_env", 12, 150, {}, {}),
    "tile12": ("formation_hd_env", 12, 200, {}, dict(force_tile_kernel=1)),
    "tile27_rows": ("formation_hd_env", 27, 40, {}, dict(force_tile_kernel=1, row_chunks=0)),
    "tile81": ("formation_hd_env", 81, 9, {}, dict(force_tile_kernel=1)),
    "tile9_flat": ("formation_hd_env", 9, 300, {}, dict(force_tile_kernel=1, no_tile_image=1)),
    "comm9": ("formation_hd_env", 9, 70, dict(silent=False), {}),
    "comm27": ("formation_hd_env", 27, 20, dict(silent=False), {}),
    "basic5_comm": ("basic_formation_env", 5, 301, dict(silent=False), {}),
    "bank9": ("formation_hd_env", 9, 1000, dict(bank=True), {}),
}


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("case", list(CASES))
def test_decode_is_bit_exact(case, dtype):
    scn, N, E, kw, opts = CASES[case]
    how = "step" if kw.get("silent", True) is False else "random"
    with nat.options(**opts):
        env = _make(scn, E, N, dtype, **kw)
        buf, want, valid = _record(env, 2 * EP + 1, how)
        _check_decode(env, buf, want, valid)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("N,n,E", [(3, 3, 1001), (9, 3, 300), (16, 4, 65)], ids=["fused3", "two_kernel9", "fused16"])
def test_decode_after_step_bfs(N, n, E, dtype):
    env = _make("formation_hd_env", E, N, dtype)
    buf, want, valid = _record(env, 2 * EP + 1, "bfs", n_layer=n)
    _check_decode(env, buf, want, valid)


# ------------------------------------------------------------------ 2. out-of-range rows
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("case", ["hd9_std", "hd27_std", "tile27_rows", "tile81", "tile9_flat", "comm27", "basic3",
                                  "partial4", "range4", "obs_env4"])
def test_out_of_range_rows_are_nan(case, dtype):
    scn, N, E, kw, opts = CASES[case]
    how = "step" if kw.get("silent", True) is False else "random"
    with nat.options(**opts):
        env = _make(scn, E, N, dtype, **kw)
        buf, want, valid = _record(env, EP + 1, how)
        R = buf.num_records
        g = torch.Generator(device=env.device).manual_seed(1)
        rows = valid[torch.randint(0, valid.shape[0], (997,), device=env.device, generator=g)]
        bad = torch.tensor([-1, R, 2 ** 40, -(2 ** 62)], device=env.device)
        pos = torch.tensor([0, 1, 100, 350, 996])              # first slot, inside tiles, last slot
        mixed = rows.clone()
        mixed[pos[:4].to(env.device)] = bad
        mixed[996] = R + 7
        ref = env.gather_observations(buf.states, rows)
        got = env.gather_observations(buf.states, mixed)
        torch.cuda.synchronize()
        miss = torch.zeros(997, dtype=torch.bool)
        miss[pos] = True
        assert torch.isnan(got[miss.to(env.device)]).all()
        assert torch.equal(got[~miss.to(env.device)], ref[~miss.to(env.device)])
        assert torch.equal(ref, want[rows])


# ------------------------------------------------------------------ 3. 64-bit record addressing
def test_records_past_four_gib():
    """fp32 hd N = 9, R = 6e7 records: pos alone spans 4.32 GB, so the records near the end lie past 2^32 bytes.  Their
    rows equal fg_obs_reward of a small env holding copies of them."""
    R, N = 60_000_000, 9
    dev = torch.device("cuda", torch.cuda.current_device())
    st = {"pos": torch.empty(R, N, 2, device=dev), "vel": torch.empty(R, N, 2, device=dev),
          "ideal_shape": torch.empty(R, N, 2, device=dev), "ideal_vel": torch.empty(R, 2, device=dev)}
    assert st["pos"].numel() * 4 > 2 ** 32
    edge = (2 ** 32) // (N * 2 * 4)                          # first record whose pos lies past 2^32 bytes
    picks = torch.cat([torch.arange(R - 600, R), torch.arange(edge - 200, edge + 200), torch.arange(0, 100)]).to(dev)
    g = torch.Generator(device=dev).manual_seed(9)
    for k, v in st.items():
        v[picks] = (torch.rand(v[picks].shape, device=dev, generator=g) * 2 - 1) * 0.5
    rows = picks[torch.randperm(picks.shape[0], device=dev, generator=g)]
    rows = torch.cat([rows, rows[:333]])                     # repeats
    env = BatchedFormationEnv("formation_hd_env", rows.shape[0], N, EP, device=dev)
    got = env.gather_observations(st, rows)
    for k, v in st.items():
        getattr(env, k).copy_(v[rows])
    env.observe()
    torch.cuda.synchronize()
    assert torch.equal(got, env.obs)
    del st


# ------------------------------------------------------------------ 4. buffer semantics
class _Model:
    """Host model of the buffer: slot -> what was written, with a version per write."""

    def __init__(self, T):
        self.T, self.slots, self.version, self.head, self.next = T, [None] * T, 0, None, 0

    def write(self, obs, tr=None):
        j = self.next
        self.version += 1
        self.slots[j] = dict(obs=obs, version=self.version, tr=None if tr is None else dict(tr, prev=self.head))
        self.head = (j, self.version)
        self.next = (j + 1) % self.T
        return j

    def valid(self):
        out = {}
        for j, s in enumerate(self.slots):
            if s is None or s["tr"] is None:
                continue
            pj, pv = s["tr"]["prev"]
            if self.slots[pj]["version"] == pv:
                out[j] = pj
        return out


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("how", ["step", "random", "bfs"])
def test_buffer_transitions(how, dtype):
    E, N, T = 16, 9, 7
    env = _make("formation_hd_env", E, N, dtype)
    buf = StateReplayBuffer(env, T)
    model = _Model(T)
    with pytest.raises(ValueError, match="mark_start"):
        buf.add(env.actions)
    with pytest.raises(ValueError, match="no transition"):
        buf.sample(4)
    buf.mark_start()
    model.write(_h(env.obs).copy())
    steps = 0

    def check():
        torch.cuda.synchronize()
        valid = model.valid()
        assert len(buf) == len(valid) * E
        g = torch.Generator(device=env.device).manual_seed(11)
        smp = buf.sample(40000, generator=g)
        g2 = torch.Generator(device=env.device).manual_seed(11)
        smp2 = buf.sample(40000, generator=g2)
        for k in smp:                                     # seeded: reproducible
            assert torch.equal(smp[k], smp2[k]), k
        slot, e = _h(smp["slot"]), _h(smp["env_index"])
        assert set(zip(slot.tolist(), e.tolist())) == {(j, x) for j in valid for x in range(E)}   # all drawn
        obs, nobs = _h(smp["obs"]), _h(smp["next_obs"])
        act, rew, done = _h(smp["actions"]), _h(smp["reward"]), _h(smp["done"])
        for j, pj in valid.items():
            sel = slot == j
            tr, ee = model.slots[j]["tr"], e[sel]
            assert np.array_equal(obs[sel], model.slots[pj]["obs"][ee])
            nxt = np.where(tr["done"][ee][:, None, None], tr["final"][ee], model.slots[j]["obs"][ee])
            assert np.array_equal(nobs[sel], nxt)
            assert np.array_equal(act[sel], tr["act"][ee])
            assert np.array_equal(rew[sel], tr["rew"][ee])
            assert np.array_equal(done[sel], tr["done"][ee])

    def advance(n):
        nonlocal steps
        for _ in range(n):
            a = _step(env, how, steps)
            buf.add(a)
            torch.cuda.synchronize()
            model.write(_h(env.obs).copy(), dict(act=_h(a).copy(), rew=_h(env.reward)[..., 0].copy(),
                                                 done=_h(env.done)[:, 0].copy(),
                                                 final=_h(env.final_observation()).copy()))
            steps += 1

    advance(EP + 1)                                        # one episode ends (terminal states in use)
    assert any(s["tr"] is not None and s["tr"]["done"].all() for s in model.slots if s)
    check()
    mask = torch.zeros(E, dtype=torch.bool, device=env.device)
    mask[::3] = True
    env.reset(mask)
    buf.mark_start()                                       # a new chain: nothing spans the reset
    model.write(_h(env.obs).copy())
    advance(3)
    check()
    advance(2 * T + 1)                                     # the ring wraps twice
    check()
    assert len(buf) == (T - 1) * E


def test_sample_shapes_and_errors():
    env = _make("formation_hd_env", 8, 3, torch.float32)
    buf = StateReplayBuffer(env, 3)
    buf.mark_start()
    env.step_random(record_actions=True)
    buf.add(env.actions)
    with pytest.raises(ValueError, match="batch_size"):
        buf.sample(0)
    with pytest.raises(ValueError, match="actions must have shape"):
        buf.add(env.actions[:, :2])
    smp = buf.sample(5)
    assert smp["obs"].shape == smp["next_obs"].shape == (5, 3, env.D)
    assert smp["actions"].shape == (5, 3, 2) and smp["reward"].shape == (5, 3) and smp["done"].dtype == torch.bool
    assert smp["env_index"].dtype == smp["slot"].dtype == torch.int64
    assert len(buf) == 8


# ------------------------------------------------------------------ 5. no side effects
OUTPUTS = ("pos", "vel", "comm", "obs", "reward", "indiv", "done", "step_count", "ep_return", "ep_collisions",
           "nan_flag", "ideal_shape", "ideal_vel", "landmarks", "landmark_vel", "actions", "final_pos", "final_vel",
           "final_ideal_shape", "final_ideal_vel", "final_landmarks")


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N", [("formation_hd_env", 9), ("formation_hd_obs_env", 4)])
def test_buffer_changes_nothing(scn, N, dtype):
    E = 300
    A = _make(scn, E, N, dtype)
    C_ = _make(scn, E, N, dtype)
    buf = StateReplayBuffer(A, 5)
    buf.mark_start()
    for s in range(3 * EP + 1):
        how = "step" if s % 2 else "random"
        buf.add(_step(A, how, s))
        buf.sample(257)
        _step(C_, how, s)
        torch.cuda.synchronize()
        for k in OUTPUTS:
            a, c = getattr(A, k), getattr(C_, k)
            if a is None:
                assert c is None
                continue
            assert torch.equal(a, c), (s, k)
        assert torch.equal(A.stats[[0, 3]], C_.stats[[0, 3]])
