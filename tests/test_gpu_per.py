"""Prioritized replay on the device (fg_per_*, PrioritizedStateReplayBuffer): the sum/min tree equals the host butterfly
reduction of its leaves bit for bit after every buffer operation, the leaves follow the update rules, sampling is the
host inverse CDF and never returns a zero leaf, sampled transitions decode like the base class's, the weights are
(min p / p)^beta, leaf offsets past 2^32 bytes work, and a buffer changes nothing the env computes."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from formation_gym import PrioritizedStateReplayBuffer  # noqa: E402
from formation_gym import _native as nat  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402

DTYPES = [torch.float32, torch.float64]
DT_IDS = ["f32", "f64"]
SCNS = [("formation_hd_env", 9), ("formation_hd_obs_env", 4)]
SCN_IDS = ["hd9", "obs_env4"]
EP = 4
LO, HI = 2.0 ** -1022, 2.0 ** 960


def _h(x):
    return x.cpu().numpy()


def _make(scn, E, N, dtype, seed=21):
    env = BatchedFormationEnv(scn, E, N, EP, dtype=dtype, seed=seed, auto_reset=True, record_final=True)
    env.reset()
    env.pos.mul_(0.3)                                      # dense: contacts, collisions, and NaN states (nan_flag)
    env.observe()
    return env


def _step(env, how, s):
    """One step; returns a copy of the actions it ran on."""
    if how == "step":
        env.sample_actions()
        env.step(env.actions)
        return env.actions.clone()
    if how == "random":
        env.step_random(record_actions=True)
        return env.actions.clone()
    act = env.actions.clone() if env._bfs_primed == 3 else env.bfs_actions(3).clone()
    env.step_bfs(3)
    return act


def host_levels(leaf):
    """[(sum, min)] of levels 1 .. depth: butterfly sums of 32 zero-padded children, min over the nonzero leaves."""
    s, m, out = leaf.astype(np.float64), np.where(leaf > 0, leaf, np.inf).astype(np.float64), []
    lane = np.arange(32)
    while True:
        n = -(-s.shape[0] // 32)
        s = np.concatenate([s, np.zeros(n * 32 - s.shape[0])]).reshape(n, 32)
        m = np.concatenate([m, np.full(n * 32 - m.shape[0], np.inf)]).reshape(n, 32)
        for off in (16, 8, 4, 2, 1):
            s = s + s[:, lane ^ off]
        s, m = s[:, 0].copy(), m.min(axis=1)
        out.append((s, m))
        if n == 1:
            return out


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.int64)


def check_tree(leaf, tsum, tmin):
    lv = host_levels(leaf)
    assert np.array_equal(_bits(np.concatenate([s for s, _ in lv])), _bits(tsum))
    assert np.array_equal(_bits(np.concatenate([m for _, m in lv])), _bits(tmin))


def _prio(td, alpha, eps):
    return np.clip((np.abs(td.astype(np.float64)) + eps) ** alpha, LO, HI)


class Sim:
    """Host model of the leaves and max_leaf under the update rules."""

    def __init__(self, buf):
        self.buf, self.leaf, self.max_leaf = buf, np.zeros((buf.capacity, buf.env.E)), 1.0

    def wrote(self, valid):
        buf = self.buf
        self.leaf[buf._head] = self.max_leaf if valid else 0.0
        for j in range(buf.capacity):
            if j not in buf._valid:
                self.leaf[j] = 0.0

    def update(self, batch, td):
        buf, E = self.buf, self.buf.env.E
        idx, st, td = _h(batch["index"]), _h(batch["stamp"]), _h(td)
        flat = self.leaf.reshape(-1)
        written = {}                                       # leaf -> value of its last applied entry
        for b in range(idx.shape[0]):
            j = idx[b]
            if np.isfinite(td[b]) and flat[j] > 0 and buf._stamp[j // E] == st[b]:
                written[j] = _prio(td[b:b + 1], buf.alpha, buf.eps)[0]
        for j, v in written.items():                       # only the winners' values reach a leaf and max_leaf
            flat[j] = v
            self.max_leaf = max(self.max_leaf, v)

    def check(self):
        buf = self.buf
        torch.cuda.synchronize()
        leaf = _h(buf._leaf)
        check_tree(leaf, _h(buf._sum), _h(buf._min))
        pos = leaf.reshape(buf.capacity, -1) > 0
        for j in range(buf.capacity):
            assert pos[j].all() if j in buf._valid else not pos[j].any(), j
        want = self.leaf.reshape(-1)
        assert np.all(np.abs(leaf - want) <= 2 * np.spacing(want)), np.abs(leaf - want).max()
        assert abs(_h(buf._max_leaf)[0] - self.max_leaf) <= 2 * np.spacing(self.max_leaf)


def _td(batch, rng, dtype):
    """Errors with NaN, inf, zeros and duplicates of one transition (the later entries must win)."""
    B = batch["index"].shape[0]
    td = rng.normal(0, 3, B)
    td[rng.choice(B, B // 8, replace=False)] = 0.0
    td[1], td[2], td[3] = np.nan, np.inf, -np.inf
    batch["index"][B // 2:B // 2 + 6] = batch["index"][0]
    batch["stamp"][B // 2:B // 2 + 6] = batch["stamp"][0]
    return torch.tensor(td, dtype=dtype, device=batch["index"].device)


# ------------------------------------------------------------------ 1. tree invariant under a random script
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N", SCNS, ids=SCN_IDS)
def test_tree_invariant(scn, N, dtype):
    E, T = 40, 5
    env = _make(scn, E, N, dtype)
    buf = PrioritizedStateReplayBuffer(env, T, alpha=0.7, eps=1e-3)
    sim = Sim(buf)
    rng = np.random.default_rng(4)
    g = torch.Generator(device=env.device).manual_seed(2)
    hows = ["step", "random"] + (["bfs"] if scn == "formation_hd_env" else [])
    buf.mark_start()
    sim.wrote(False)
    sim.check()
    old, steps = [], 0
    for op in range(60):
        r = rng.random()
        if r < 0.45 or not buf._valid:
            buf.add(_step(env, hows[steps % len(hows)], steps))
            steps += 1
            sim.wrote(True)
        elif r < 0.55:
            mask = torch.tensor(rng.random(E) < 0.3, device=env.device)
            env.reset(mask)
            buf.mark_start()
            sim.wrote(False)
        elif r < 0.85:
            b = buf.sample(64, beta=0.5, generator=g)
            td = _td(b, rng, torch.float32 if op % 2 else torch.float64)
            buf.update_priorities(b, td)
            sim.update(b, td)
            old.append(b)
        else:                                              # a batch sampled before slots were overwritten / dropped
            b = old[rng.integers(len(old))] if old else buf.sample(64, generator=g)
            td = torch.tensor(rng.normal(0, 10, 64), dtype=torch.float64, device=env.device)
            buf.update_priorities(b, td)
            sim.update(b, td)
        sim.check()
    assert steps > 2 * T and sim.max_leaf > 1.0


# ------------------------------------------------------------------ 2. sampling = host inverse CDF; 4. decoding
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N", SCNS, ids=SCN_IDS)
def test_sampling_and_decoding(scn, N, dtype):
    E, T = 64, 6
    env = _make(scn, E, N, dtype)
    buf = PrioritizedStateReplayBuffer(env, T)
    rng = np.random.default_rng(7)
    S, F, A, R, D = {}, {}, {}, {}, {}
    buf.mark_start()
    S[buf._head] = _h(env.obs).copy()
    for s in range(2 * T + 3):                             # wraps; episodes end (terminal rows in use)
        a = _step(env, "random" if s % 2 else "step", s)
        buf.add(a)
        j = buf._head
        S[j], F[j], A[j] = _h(env.obs).copy(), _h(env.final_observation()).copy(), _h(a).copy()
        R[j], D[j] = _h(env.reward)[..., 0].copy(), _h(env.done)[:, 0].copy()
        if s % 3 == 2:
            b = buf.sample(256)
            buf.update_priorities(b, torch.tensor(rng.lognormal(0, 2, 256), device=env.device))
    assert any(D[j].any() for j in buf._valid)
    B = 8192
    b = buf.sample(B, beta=0.4, generator=torch.Generator(device=env.device).manual_seed(13))
    u = _h(torch.rand(B, dtype=torch.float64, generator=torch.Generator(device=env.device).manual_seed(13),
                      device=env.device))
    torch.cuda.synchronize()
    leaf = _h(buf._leaf)
    total = _h(buf._sum)[-1]
    cum = np.cumsum(leaf)
    x = u * total
    want = np.searchsorted(cum, x, "right")
    lo = np.where(want > 0, cum[np.maximum(want - 1, 0)], 0.0)
    far = (np.abs(x - lo) > 1e-12 * total) & (np.abs(cum[np.minimum(want, cum.size - 1)] - x) > 1e-12 * total)
    idx = _h(b["index"])
    assert far.mean() > 0.99
    assert np.array_equal(idx[far], want[far])
    assert (leaf[idx] > 0).all()
    slot, e = _h(b["slot"]), _h(b["env_index"])
    assert np.array_equal(slot * E + e, idx)
    st = np.array(buf._stamp)
    assert np.array_equal(_h(b["stamp"]), st[slot])
    prev = np.array([buf._valid[j] for j in slot])
    done = _h(b["done"])
    ob, nob = _h(b["obs"]), _h(b["next_obs"])
    for k in range(B):
        j, x_, p = slot[k], e[k], prev[k]
        assert np.array_equal(ob[k], S[p][x_], equal_nan=True)
        nxt = F[j][x_] if D[j][x_] else S[j][x_]
        assert np.array_equal(nob[k], nxt, equal_nan=True)
        assert done[k] == D[j][x_]
    assert np.array_equal(_h(b["actions"]), np.stack([A[j][x_] for j, x_ in zip(slot, e)]))
    assert np.array_equal(_h(b["reward"]), np.stack([R[j][x_] for j, x_ in zip(slot, e)]))
    # the record rows fg_per_sample hands to fg_obs_gather are the base class's
    rows = env.gather_observations(buf.states, torch.tensor(np.concatenate([prev * E + e, np.where(
        done, slot * E + e + T * E, slot * E + e)]), device=env.device))
    assert torch.equal(torch.cat([b["obs"], b["next_obs"]]).isnan(), rows.isnan())
    assert torch.equal(torch.nan_to_num(torch.cat([b["obs"], b["next_obs"]])), torch.nan_to_num(rows))
    # 5. weights
    w = (_h(buf._min)[-1] / leaf[idx]) ** 0.4
    got = _h(b["weights"]).astype(np.float64)
    assert np.allclose(got, w, rtol=1e-12 if dtype == torch.float64 else 1e-6, atol=0)
    assert got.max() <= 1.0
    b0 = buf.sample(1000, beta=0.0)
    assert torch.equal(b0["weights"], torch.ones_like(b0["weights"]))
    # 7. the same seed gives the same samples
    g1, g2 = (torch.Generator(device=env.device).manual_seed(5) for _ in range(2))
    s1, s2 = buf.sample(3000, 0.6, g1), buf.sample(3000, 0.6, g2)
    for k in s1:
        x, y = s1[k], s2[k]
        assert torch.equal(x.nan_to_num(), y.nan_to_num()) if x.is_floating_point() else torch.equal(x, y), k


# ------------------------------------------------------------------ 3. zero leaves are never returned
def _raw_tree(T, E, leaf=None):
    dev = torch.device("cuda", torch.cuda.current_device())
    nodes, depth, scratch = C.c_longlong(), C.c_int(), C.c_longlong()
    lib = nat.load()
    nat.check(lib.fg_per_layout(T, E, C.byref(nodes), C.byref(depth), C.byref(scratch)), "fg_per_layout")
    kw = dict(device=dev, dtype=torch.float64)
    a = dict(leaf=torch.zeros(T * E, **kw) if leaf is None else leaf, sum=torch.zeros(nodes.value, **kw),
             min=torch.full((nodes.value,), float("inf"), **kw), max_leaf=torch.ones(1, **kw),
             stamp=torch.zeros(T, dtype=torch.int64, device=dev), prev=torch.full((T,), -1, dtype=torch.int64, device=dev),
             scratch=torch.zeros(scratch.value // 4, dtype=torch.int32, device=dev))
    t = nat.fg_per()
    for k, v in a.items():
        setattr(t, k, v.data_ptr())
    t.slots, t.envs = T, E
    return lib, t, a


def _raw_sample(lib, t, a, u, N=1, A=1):
    dev, B = u.device, u.shape[0]
    M = t.slots * t.envs
    done = torch.zeros(M, dtype=torch.uint8, device=dev)
    act = torch.zeros(M, N, A, device=dev)
    rew = torch.zeros(M, N, device=dev)
    ids = torch.empty(6, B, dtype=torch.int64, device=dev)
    o = dict(done=torch.empty(B, dtype=torch.uint8, device=dev), w=torch.empty(B, device=dev),
             act=torch.empty(B, N, A, device=dev), rew=torch.empty(B, N, device=dev))
    nat.check(lib.fg_per_sample(C.byref(t), u.data_ptr(), B, 0.5, done.data_ptr(), act.data_ptr(), rew.data_ptr(), N, A,
                                ids[0].data_ptr(), ids[2].data_ptr(), ids[3].data_ptr(), ids[4].data_ptr(),
                                ids[5].data_ptr(), o["done"].data_ptr(), o["w"].data_ptr(), o["act"].data_ptr(),
                                o["rew"].data_ptr(), None), "fg_per_sample")
    torch.cuda.synchronize()
    return ids, o


def test_zero_leaves_are_never_returned():
    T, E = 3, 1111                                         # M = 3333, not a multiple of 32; depth 3
    M = T * E
    rng = np.random.default_rng(0)
    leaf = np.zeros(M)
    nz = np.sort(rng.choice(M, 40, replace=False))
    leaf[nz] = rng.lognormal(0, 3, nz.size)
    leaf[nz[:5]] = LO
    leaf[nz[5:10]] = HI
    leaf[nz[10]], leaf[nz[10] + 1] = LO, HI                # 2^-1022 next to 2^960
    leaf[M - 1] = LO                                       # the last leaf, in a part-filled group of 32
    leaf[0] = 0.0
    dev = torch.device("cuda", torch.cuda.current_device())
    lib, t, a = _raw_tree(T, E, torch.tensor(leaf, device=dev))
    lv = host_levels(leaf)
    a["sum"].copy_(torch.tensor(np.concatenate([s for s, _ in lv])))
    a["min"].copy_(torch.tensor(np.concatenate([m for _, m in lv])))
    total = lv[-1][0][0]
    cum = np.cumsum(leaf)
    u = np.concatenate([[0.0, 1.0 - 2.0 ** -53, np.nextafter(1.0, 0) * 0.5], cum / total,
                        np.nextafter(cum / total, 0), rng.random(20000)])
    u = u[(u >= 0) & (u < 1)]
    ids, o = _raw_sample(lib, t, a, torch.tensor(u, device=dev))
    idx = _h(ids[2])
    assert (idx >= 0).all() and (idx < M).all()
    assert (leaf[idx] > 0).all()
    # a tree of zeros only: every draw reports -1 and NaN
    lib, t, a = _raw_tree(1, 70)
    ids, o = _raw_sample(lib, t, a, torch.rand(50, dtype=torch.float64, device=dev))
    assert (_h(ids) == -1).all() and torch.isnan(o["w"]).all() and torch.isnan(o["act"]).all()


# ------------------------------------------------------------------ 5. alpha = 0: uniform over the valid transitions
def test_alpha_zero_is_uniform():
    from scipy.stats import chi2
    E, T = 16, 5
    env = _make("formation_hd_env", E, 3, torch.float32)
    buf = PrioritizedStateReplayBuffer(env, T, alpha=0.0)
    buf.mark_start()
    rng = np.random.default_rng(1)
    for s in range(T + 2):
        buf.add(_step(env, "random", s))
        b = buf.sample(128)
        buf.update_priorities(b, torch.tensor(rng.normal(0, 5, 128), device=env.device))
    torch.cuda.synchronize()
    leaf = _h(buf.priorities)
    valid = sorted(buf._valid)
    assert np.array_equal(leaf[valid], np.ones((len(valid), E)))
    n = 1 << 20
    b = buf.sample(n, beta=0.4, generator=torch.Generator(device=env.device).manual_seed(3))
    assert torch.equal(b["weights"], torch.ones_like(b["weights"]))
    counts = np.bincount(_h(b["index"]), minlength=T * E).reshape(T, E)
    assert counts[[j for j in range(T) if j not in buf._valid]].sum() == 0
    obs = counts[valid].reshape(-1)
    k = obs.size
    stat = ((obs - n / k) ** 2 / (n / k)).sum()
    assert stat < chi2.ppf(1 - 1e-6, k - 1), (stat, k)


# ------------------------------------------------------------------ 6. leaf byte offsets past 2^32
def test_large_index_space():
    """3 slots x (2^28 + 5) envs: M > 2^29 leaves, 6.4 GB of leaves, slot 2's past 2^32 bytes."""
    T, E = 3, (1 << 28) + 5
    M = T * E
    assert M > 1 << 29 and 2 * E * 8 > 1 << 32
    lib, t, a = _raw_tree(T, E)
    dev = a["leaf"].device
    nat.check(lib.fg_per_fill(C.byref(t), 1, -1, 1, 0, -1, None), "fg_per_fill")
    nat.check(lib.fg_per_fill(C.byref(t), 2, 1, 2, 1, -1, None), "fg_per_fill")
    hi = [2 * E, 2 * E + (1 << 27), M - 1]                 # 1e9 each; alpha = 1 and integer |td| + eps: exact sums
    idx = torch.tensor(hi + [M - 2, M - 2, M - 3, E + 7], dtype=torch.int64, device=dev)
    st = torch.tensor([2, 2, 2, 2, 2, 1, 1], dtype=torch.int64, device=dev)   # M - 3: stale stamp; E + 7: a zero leaf
    td = torch.tensor([1e9 - 0.5] * 3 + [10.5, -6.5, 99.5, 99.5], dtype=torch.float64, device=dev)
    nat.check(lib.fg_per_update(C.byref(t), idx.data_ptr(), st.data_ptr(), td.data_ptr(), 1, idx.shape[0], 1.0, 0.5,
                                None), "fg_per_update")
    torch.cuda.synchronize()
    lf = a["leaf"]
    assert np.allclose(_h(lf[idx]), [1e9] * 3 + [7.0, 7.0, 1.0, 0.0], rtol=1e-15, atol=0)   # the later duplicate wins
    assert float(lf[:2 * E].sum()) == 0.0
    total = (E - 4) + 3e9 + 7.0
    assert abs(float(a["sum"][-1]) - total) <= 1e-12 * total and float(a["min"][-1]) == 1.0
    assert abs(float(a["max_leaf"][0]) - 1e9) <= 1e-6
    nodes, depth, sc = C.c_longlong(), C.c_int(), C.c_longlong()
    lib.fg_per_layout(T, E, C.byref(nodes), C.byref(depth), C.byref(sc))
    cnt, off, n = [M], [0, 0], M
    for k in range(1, depth.value + 1):
        n = -(-n // 32)
        cnt.append(n)
        off.append(off[-1] + n)
    lane = np.arange(32)
    for j in hi + [M - 2, M - 3]:                          # every ancestor of the updated leaves, against the host
        for k in range(1, depth.value + 1):
            node = j >> (5 * k)
            lo_c, hi_c = node * 32, min(node * 32 + 32, cnt[k - 1])
            ch = np.zeros(32)
            ch[:hi_c - lo_c] = _h(lf[lo_c:hi_c] if k == 1 else a["sum"][off[k - 1] + lo_c:off[k - 1] + hi_c])
            for o in (16, 8, 4, 2, 1):
                ch = ch + ch[lane ^ o]
            assert _bits(_h(a["sum"][off[k] + node:off[k] + node + 1])) == _bits(ch[:1]), (j, k)
    u = torch.tensor([1e-9, 0.5, 1.0 - 1e-4, 1.0 - 2.0 ** -53], dtype=torch.float64, device=dev)
    ids, o = _raw_sample(lib, t, a, u)
    assert _h(ids[2]).tolist() == [2 * E, 2 * E + (1 << 27), M - 1, M - 1]
    assert _h(ids[4]).tolist() == [2, 2, 2, 2] and _h(ids[3]).tolist() == [2] * 4
    assert _h(ids[0]).tolist() == [E + 0, E + (1 << 27), 2 * E - 1, 2 * E - 1]
    assert np.allclose(_h(o["w"]), (1.0 / 1e9) ** 0.5, rtol=1e-6)
    del a, lf


# ------------------------------------------------------------------ 7. no side effects
OUTPUTS = ("pos", "vel", "comm", "obs", "reward", "indiv", "done", "step_count", "ep_return", "ep_collisions",
           "nan_flag", "ideal_shape", "ideal_vel", "landmarks", "landmark_vel", "actions", "final_pos", "final_vel",
           "final_ideal_shape", "final_ideal_vel", "final_landmarks")


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scn,N", SCNS, ids=SCN_IDS)
def test_buffer_changes_nothing(scn, N, dtype):
    E = 300
    A_, C_ = _make(scn, E, N, dtype), _make(scn, E, N, dtype)
    buf = PrioritizedStateReplayBuffer(A_, 5)
    buf.mark_start()
    for s in range(3 * EP + 1):
        how = "step" if s % 2 else "random"
        buf.add(_step(A_, how, s))
        b = buf.sample(257, beta=0.4)
        buf.update_priorities(b, b["reward"][:, 0].float())
        _step(C_, how, s)
        torch.cuda.synchronize()
        for k in OUTPUTS:
            a, c = getattr(A_, k), getattr(C_, k)
            if a is None:
                assert c is None
                continue
            assert torch.equal(a, c), (s, k)
