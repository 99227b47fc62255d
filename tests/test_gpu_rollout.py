"""On-policy rollouts on the device: fg_gae against a numpy loop of its recurrence, bit for bit in both precisions, and
against onpolicy's GAE; truncations bootstrapped from final_value; NaN isolation; offsets past 2^32 bytes; and
StateRolloutBuffer's decoded minibatches, bootstrapping, permutation coverage and an env that is unchanged with a buffer
attached."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from formation_gym import StateRolloutBuffer  # noqa: E402
from formation_gym import _native as nat  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402

DTYPES = [torch.float32, torch.float64]
DT_IDS = ["f32", "f64"]
NP = {torch.float32: np.float32, torch.float64: np.float64}
UINT = {torch.float32: np.uint32, torch.float64: np.uint64}
DEV = torch.device("cuda", 0)


def _h(x):
    return x.cpu().numpy()


def _bits(x, dtype):
    return np.ascontiguousarray(x).view(UINT[dtype])


def host_gae(rew, val, done, fv, gamma, lam, dt):
    """The recurrence of include/formation_gym_b200.h fg_gae in numpy, in dtype dt (every op rounded once)."""
    T = rew.shape[0]
    g, gl = dt(gamma), dt(gamma * lam)
    a = np.zeros(rew.shape[1:], dt)
    adv, ret = np.empty_like(rew), np.empty_like(rew)
    with np.errstate(all="ignore"):
        for t in range(T - 1, -1, -1):
            d = (done[t] != 0).reshape(done.shape[1], *([1] * (rew.ndim - 2)))
            nv = np.where(d, fv[t] if fv is not None else dt(0), val[t + 1])
            delta = (rew[t] + g * nv) - val[t]
            a = np.where(d, delta, delta + gl * a)
            adv[t], ret[t] = a, a + val[t]
    return adv, ret


def dev_gae(rew, val, done, fv, gamma, lam, adv=None, ret=None):
    """One fg_gae launch on device tensors; returns (adv, ret)."""
    lib = nat.load()
    T, E, N = rew.shape
    adv = torch.empty_like(rew) if adv is None else adv
    ret = torch.empty_like(rew) if ret is None else ret
    sfx = "" if rew.dtype == torch.float32 else "_f64"
    P = nat.ptr
    rc = getattr(lib, "fg_gae" + sfx)(P(rew), P(val), P(fv), P(done), P(adv), P(ret), T, E, N, gamma, lam,
                                      torch.cuda.current_stream().cuda_stream)
    nat.check(rc, "fg_gae")
    return adv, ret


def _inputs(T, E, N, dtype, pattern, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    kw = dict(device=DEV, dtype=dtype)
    rew = torch.randn(T, E, N, generator=g, **kw)
    val = torch.randn(T + 1, E, N, generator=g, **kw)
    fv = torch.randn(T, E, N, generator=g, **kw)
    t = torch.arange(T, device=DEV)[:, None]
    e = torch.arange(E, device=DEV)[None, :]
    done = {"none": torch.zeros(T, E, dtype=torch.bool, device=DEV),
            "all": torch.ones(T, E, dtype=torch.bool, device=DEV),
            "staggered": (t + e) % 4 == 3,
            "t0": (t == 0).expand(T, E),
            "tlast": (t == T - 1).expand(T, E),
            "random": torch.rand(T, E, generator=g, device=DEV) < 0.2}[pattern].to(torch.uint8).contiguous()
    return rew, val, fv, done


SHAPES = [(1, 7, 3), (5, 13, 5), (25, 37, 9), (17, 1000, 27), (3, 40000, 9)]   # (3, 40000, 9): 360000 columns
PATTERNS = ["none", "all", "staggered", "t0", "tlast", "random"]


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", SHAPES, ids=["x".join(map(str, s)) for s in SHAPES])
def test_gae_bit_exact(shape, dtype):
    T, E, N = shape
    dt = NP[dtype]
    for i, pattern in enumerate(PATTERNS):
        rew, val, fv, done = _inputs(T, E, N, dtype, pattern, seed=i)
        hr, hv, hf, hd = _h(rew), _h(val), _h(fv), _h(done)
        for final in (True, False):
            gamma, lam = (0.99, 0.95) if final else (0.97, 0.9)
            adv, ret = dev_gae(rew, val, done, fv if final else None, gamma, lam)
            wa, wr = host_gae(hr, hv, hd, hf if final else None, gamma, lam, dt)
            for got, want, what in ((adv, wa, "adv"), (ret, wr, "ret")):
                np.testing.assert_array_equal(_bits(_h(got), dtype), _bits(want, dtype),
                                              err_msg="%s %s final=%s" % (what, pattern, final))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_outputs_are_written_everywhere(dtype):
    """Whatever adv / ret held before the launch does not survive it."""
    T, E, N = 9, 301, 9
    rew, val, fv, done = _inputs(T, E, N, dtype, "random", seed=4)
    a0, r0 = dev_gae(rew, val, done, fv, 0.99, 0.95)
    a1, r1 = dev_gae(rew, val, done, fv, 0.99, 0.95, adv=torch.full_like(rew, float("nan")),
                     ret=torch.full_like(rew, float("inf")))
    assert torch.equal(a0, a1) and torch.equal(r0, r1)


def onpolicy_gae(rew, val, done, gamma, lam):
    """onpolicy SharedReplayBuffer.compute_returns (use_gae, no PopArt / ValueNorm, use_proper_time_limits=False),
    restated in torch: masks[t + 1] = 1 - done[t]."""
    T = rew.shape[0]
    masks = 1.0 - done.to(rew.dtype)[..., None]
    gae = torch.zeros_like(rew[0])
    ret = torch.empty_like(rew)
    for step in reversed(range(T)):
        delta = rew[step] + gamma * val[step + 1] * masks[step] - val[step]
        gae = delta + gamma * lam * masks[step] * gae
        ret[step] = gae + val[step]
    return ret - val[:T], ret


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("pattern", PATTERNS)
def test_null_final_value_is_onpolicy_gae(pattern, dtype):
    T, E, N = 25, 257, 9
    rew, val, fv, done = _inputs(T, E, N, dtype, pattern, seed=7)
    adv, ret = dev_gae(rew, val, done, None, 0.99, 0.95)
    wa, wr = onpolicy_gae(rew, val, done, 0.99, 0.95)
    tol = dict(rtol=1e-5, atol=1e-5) if dtype == torch.float32 else dict(rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(adv, wa, **tol)
    torch.testing.assert_close(ret, wr, **tol)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_lambda_one_is_the_discounted_return(dtype):
    T, E, N = 30, 65, 4
    rew, val, fv, done = _inputs(T, E, N, dtype, "none", seed=8)
    gamma = 0.95
    adv, ret = dev_gae(rew, val, done, fv, gamma, 1.0)
    r64, v64 = rew.double(), val.double()
    want = torch.empty_like(r64)
    acc = v64[T]
    for t in range(T - 1, -1, -1):
        acc = r64[t] + gamma * acc
        want[t] = acc
    tol = dict(rtol=1e-4, atol=1e-4) if dtype == torch.float32 else dict(rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(ret.double(), want, **tol)
    torch.testing.assert_close(adv.double(), want - v64[:T], **tol)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("final", [True, False], ids=["final", "terminal"])
def test_value_after_a_done_is_never_read(final, dtype):
    """value[t+1] of an env whose episode ended at t is V(reset state); poisoned with NaN / inf it must not reach
    adv / ret at t or before (a mask multiply would give NaN * 0 = NaN).  It is V(s_{t+1}) of the next step, so the
    steps after t do see it."""
    T, E, N = 12, 40, 9
    rew, val, fv, done = _inputs(T, E, N, dtype, "none", seed=9)
    t_end = torch.arange(E, device=DEV) % T                 # env e ends once, at t_end[e] (T-1: the bootstrap value)
    done[t_end, torch.arange(E, device=DEV)] = 1
    a0, r0 = dev_gae(rew, val, done, fv if final else None, 0.99, 0.95)
    bad = val.clone()
    poison = torch.tensor([float("nan"), float("inf"), -float("inf")], dtype=dtype, device=DEV)
    for e in range(E):
        bad[int(t_end[e]) + 1, e] = poison[e % 3]
    a1, r1 = dev_gae(rew, bad, done, fv if final else None, 0.99, 0.95)
    for e in range(E):
        upto = int(t_end[e]) + 1
        assert torch.isfinite(a1[:upto, e]).all() and torch.isfinite(r1[:upto, e]).all()
        assert torch.equal(a1[:upto, e], a0[:upto, e]) and torch.equal(r1[:upto, e], r0[:upto, e])


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_poisoned_column_stays_in_its_column(dtype):
    T, E, N = 20, 50, 9
    rew, val, fv, done = _inputs(T, E, N, dtype, "random", seed=10)
    a0, r0 = dev_gae(rew, val, done, fv, 0.99, 0.95)
    e0, n0 = 17, 4
    for arr in (rew, val, fv):
        arr[:, e0, n0] = float("nan")
    a1, r1 = dev_gae(rew, val, done, fv, 0.99, 0.95)
    keep = torch.ones(E, N, dtype=torch.bool, device=DEV)
    keep[e0, n0] = False
    assert torch.isnan(a1[:, e0, n0]).all()
    np.testing.assert_array_equal(_bits(_h(a1[:, keep]), dtype), _bits(_h(a0[:, keep]), dtype))
    np.testing.assert_array_equal(_bits(_h(r1[:, keep]), dtype), _bits(_h(r0[:, keep]), dtype))


def test_offsets_past_four_gib():
    """fp32, T = 4, 40e6 envs x 9 agents: M = 3.6e8 columns, each [T, E, N] array 5.76 GB and step 3 at 4.32 GB and
    beyond, so the elements of the last step lie past 2^32 bytes (and past 2^30 elements).  About 30 GB of device
    memory in all.  Columns at both ends and a random sample are checked bit for bit against the host loop."""
    T, E, N = 4, 40_000_000, 9
    M = E * N
    assert (T - 1) * M * 4 > 1 << 32
    g = torch.Generator(device=DEV).manual_seed(11)
    kw = dict(device=DEV, dtype=torch.float32)
    rew = torch.randn(T, E, N, generator=g, **kw)
    val = torch.randn(T + 1, E, N, generator=g, **kw)
    fv = torch.randn(T, E, N, generator=g, **kw)
    done = (torch.rand(T, E, generator=g, device=DEV) < 0.3).to(torch.uint8)
    adv, ret = dev_gae(rew, val, done, fv, 0.99, 0.95)
    cols = torch.cat([torch.arange(4096, device=DEV), torch.arange(M - 4096, M, device=DEV),
                      torch.randint(0, M, (4096,), generator=g, device=DEV)])
    pick = lambda x: _h(x.view(x.shape[0], M)[:, cols])   # noqa: E731
    envs = cols // N
    wa, wr = host_gae(pick(rew), pick(val), _h(done[:, envs]), pick(fv), 0.99, 0.95, np.float32)
    np.testing.assert_array_equal(_bits(pick(adv), torch.float32), _bits(wa, torch.float32))
    np.testing.assert_array_equal(_bits(pick(ret), torch.float32), _bits(wr, torch.float32))
    del rew, val, fv, done, adv, ret
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ StateRolloutBuffer
EP = 5


def _staggered_env(scn, E, N, dtype, seed=3, record_final=False):
    """An auto-resetting env whose episodes are staggered by reset(mask), so they end at different rollout steps."""
    env = BatchedFormationEnv(scn, E, N, EP, dtype=dtype, seed=seed, auto_reset=True, record_final=record_final)
    env.reset()
    idx = torch.arange(E, device=env.device)
    for s in range(EP):
        env.step_random()
        env.reset(mask=idx % EP == s)
    return env


def _rollout(env, buf, how, g, with_final):
    """One rollout of buf.num_steps steps; returns what every record and per-step array must hold."""
    T, E, N = buf.num_steps, env.E, env.N
    kw = dict(device=env.device, dtype=env.dtype)
    want = {k: [] for k in ("obs", "actions", "log_probs", "values", "rewards", "done", "final_values")}
    buf.start()
    for t in range(T):
        want["obs"].append(env.obs.clone())
        if how == "step":
            act = torch.rand(E, N, env.act_dim, generator=g, **kw) * 2 - 1
            env.step(act)
        else:
            env.step_random(record_actions=True)
            act = env.actions
        lp = torch.randn(E, N, generator=g, **kw)
        v = torch.randn(E, N, generator=g, device=env.device, dtype=torch.float64)   # converted by copy_
        fv = torch.randn(E, N, generator=g, **kw) if with_final else None
        want["actions"].append(act.clone())
        want["log_probs"].append(lp)
        want["values"].append(v.to(env.dtype))
        want["rewards"].append(env.reward[..., 0].clone())
        want["done"].append(env.done[:, 0].clone())
        want["final_values"].append(fv if with_final else torch.zeros(E, N, **kw))
        buf.insert(act, lp, v, final_values=fv)
    nv = torch.randn(E, N, generator=g, **kw)
    want["values"].append(nv)
    buf.compute_returns(nv, gamma=0.99, gae_lambda=0.95)
    return {k: torch.stack(v) for k, v in want.items()}


ENV_OUTPUTS = ("pos", "vel", "comm", "obs", "reward", "indiv", "done", "step_count", "ep_return", "ep_collisions",
               "nan_flag", "ideal_shape", "ideal_vel", "landmarks", "landmark_vel", "actions", "final_pos", "final_vel",
               "final_ideal_shape", "final_ideal_vel", "final_landmarks")
ROLLOUT_CASES = [("formation_hd_env", 9, 48), ("basic_formation_env", 3, 40), ("formation_hd_obs_env", 4, 36)]


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("how", ["step", "random"])
@pytest.mark.parametrize("scn,N,E", ROLLOUT_CASES, ids=[c[0] for c in ROLLOUT_CASES])
def test_minibatches_decode_the_rollout(scn, N, E, how, dtype):
    env = _staggered_env(scn, E, N, dtype)
    T = 12
    buf = StateRolloutBuffer(env, T)
    g = torch.Generator(device=env.device).manual_seed(1)
    for r in range(2):                                      # the second rollout starts where the first ended
        want = _rollout(env, buf, how, g, with_final=r == 0)
        assert want["done"].any(0).all()                    # every env ended an episode in the rollout...
        assert (want["done"].int().argmax(0) != want["done"].int().argmax(0)[0]).any()   # ...at different t
        for k in ("actions", "log_probs", "rewards", "final_values"):
            assert torch.equal(getattr(buf, k), want[k]), k
        assert torch.equal(buf.values, want["values"]) and torch.equal(buf.done, want["done"])
        wa, wr = host_gae(_h(want["rewards"]), _h(want["values"]), _h(want["done"]), _h(want["final_values"]),
                          0.99, 0.95, NP[dtype])
        assert np.array_equal(_bits(_h(buf.advantages), dtype), _bits(wa, dtype))
        assert np.array_equal(_bits(_h(buf.returns), dtype), _bits(wr, dtype))
        seen = []
        for mb in buf.minibatches(5, generator=g):
            t, e = mb["step_index"], mb["env_index"]
            B = t.shape[0]
            assert B == (T * E) // 5 and mb["obs"].shape == (B, N, env.D)
            assert torch.equal(mb["obs"], want["obs"][t, e])    # bit-identical to what the env returned
            assert torch.equal(mb["share_obs"], want["obs"].view(T, E, N * env.D)[t, e])
            assert mb["share_obs"].data_ptr() == mb["obs"].data_ptr()
            assert torch.equal(mb["actions"], want["actions"][t, e])
            assert torch.equal(mb["log_probs"], want["log_probs"][t, e])
            assert torch.equal(mb["values"], want["values"][t, e])
            assert torch.equal(mb["returns"], buf.returns[t, e])
            assert torch.equal(mb["advantages"], buf.advantages[t, e])
            seen.append(t * E + e)
        seen = torch.cat(seen)
        assert seen.unique().numel() == seen.numel() == 5 * ((T * E) // 5)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_bootstrapping_from_final_observation(dtype):
    """A critic of the observation (here a fixed linear map) gives V(s_t) and, through final_observation(), V of the
    state each episode ended in; returns equal the host recurrence fed the same values, and without final_values the
    terminal variant.  The two differ where an episode ended."""
    E, N, T = 64, 9, 11
    w = None
    critic = lambda o: o @ w                                # noqa: E731  [E,N,D] -> [E,N]
    res = {}
    for with_final in (True, False):
        twin = _staggered_env("formation_hd_env", E, N, dtype, record_final=True)
        if w is None:
            w = torch.linspace(-1, 1, twin.D, device=twin.device, dtype=dtype)
        buf = StateRolloutBuffer(twin, T)
        buf.start()
        rew, val, done, fvs = [], [], [], []
        for t in range(T):
            v = critic(twin.obs)
            twin.step_random(record_actions=True)
            fv = critic(twin.final_observation())
            buf.insert(twin.actions, torch.zeros(E, N, device=twin.device, dtype=dtype), v,
                       final_values=fv if with_final else None)
            rew.append(twin.reward[..., 0].clone())
            val.append(v)
            done.append(twin.done[:, 0].clone())
            fvs.append(fv)
        nv = critic(twin.obs)
        buf.compute_returns(nv, 0.99, 0.95)
        val.append(nv)
        wa, wr = host_gae(_h(torch.stack(rew)), _h(torch.stack(val)), _h(torch.stack(done)),
                          _h(torch.stack(fvs)) if with_final else None, 0.99, 0.95, NP[dtype])
        assert np.array_equal(_bits(_h(buf.returns), dtype), _bits(wr, dtype))
        assert np.array_equal(_bits(_h(buf.advantages), dtype), _bits(wa, dtype))
        res[with_final] = (buf.returns.clone(), torch.stack(done))
    d = res[True][1]
    assert d.any()
    ended = d[:, :, None].expand(T, E, N)
    assert not torch.equal(res[True][0][ended], res[False][0][ended])


def test_minibatch_coverage_and_seeds():
    E, N, T = 30, 9, 7                                     # T * E = 210
    env = _staggered_env("formation_hd_env", E, N, torch.float32)
    buf = StateRolloutBuffer(env, T)
    g = torch.Generator(device=env.device).manual_seed(2)
    _rollout(env, buf, "random", g, with_final=False)
    for n in (1, 3, 7, 210):                               # divisors: every (t, e) exactly once per epoch
        for _ in range(2):
            rows = torch.cat([mb["step_index"] * E + mb["env_index"] for mb in buf.minibatches(n, generator=g)])
            assert torch.equal(rows.sort().values, torch.arange(T * E, device=env.device))
    for n in (4, 11, 209):                                 # not divisors: the remainder is dropped
        mbs = list(buf.minibatches(n, generator=g))
        assert len(mbs) == n and all(mb["obs"].shape[0] == (T * E) // n for mb in mbs)
        rows = torch.cat([mb["step_index"] * E + mb["env_index"] for mb in mbs])
        assert rows.numel() == n * ((T * E) // n) and rows.unique().numel() == rows.numel()
    runs = []
    for _ in range(2):
        gg = torch.Generator(device=env.device).manual_seed(123)
        runs.append([(mb["step_index"], mb["env_index"], mb["obs"]) for mb in buf.minibatches(4, generator=gg)])
    for a, b in zip(*runs):
        assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("scn,N", [("formation_hd_env", 9), ("basic_formation_env", 3)])
def test_buffer_changes_nothing(scn, N):
    E, T = 64, 6
    envs = [_staggered_env(scn, E, N, torch.float32, record_final=True) for _ in range(2)]
    buf = StateRolloutBuffer(envs[0], T)
    g = torch.Generator(device=envs[0].device).manual_seed(5)
    for r in range(3):
        buf.start()
        for t in range(T):
            for env in envs:
                env.step_random(record_actions=True)
            fv = envs[0].final_observation().sum(-1)
            buf.insert(envs[0].actions, torch.zeros(E, N, device=envs[0].device), fv, final_values=fv)
            for k in ENV_OUTPUTS:
                a, b = getattr(envs[0], k), getattr(envs[1], k)
                assert (a is None and b is None) or torch.equal(a, b), (r, t, k)
        buf.compute_returns(torch.zeros(E, N, device=envs[0].device))
        for _ in buf.minibatches(3, generator=g):
            pass
    # stats = (episodes, return sum, return sum of squares, collisions): the kernels add each CTA's partial sums with
    # fp64 atomicAdd, so the two real-valued sums depend on the CTAs' order in the last bits, with or without a buffer
    # (test_gpu_replay.py compares the same two integer-valued entries)
    s0, s1 = envs[0].stats, envs[1].stats
    assert torch.equal(s0[[0, 3]], s1[[0, 3]])
    torch.testing.assert_close(s0[[1, 2]], s1[[1, 2]], rtol=1e-12, atol=0.0)
