"""Edge states against the numpy oracle, on every step kernel: non-finite state, distances exactly on a decision
threshold, and exact ties in the controller's argsort / argmin.

Random batches almost never land on these inputs, and the kernel-vs-kernel tests cannot see a rule that all kernels
share.  Each test here picks its kernel path with the ``nat.options`` switches and the dispatch rules of
fg_abi_impl.cuh (warp_path_ok / lm_warp_ok / launch_warp):

  k_hd_warp STD fp32 .... formation_hd_env, fp32, default step, N in {3, 4, 8, 9, 16, 25, 27, 32}
  k_hd_warp generic ..... the same N with no_std_kernel = 1 (fp32) or fp64, with and without observations
  k_hd_warp basic ....... basic_formation_env, N = L = 3
  k_hd_warp + policy .... step_bfs(3) at N = 9, step_bfs(2) at N = 4
  k_step scalar pairs ... force_tile_kernel = 1 at N = 9; N = 10; N = 81 with no_fast_pairs = 1
  k_step HET ............ per-agent masses
  k_step packed pairs ... fp32, N in {40, 243} without observations (cell lists and no_cells = 1); N = 81 with them
  k_lm_warp ............. partial N = 4, partial_range N = 5, obstacle N = 4
  k_step_obst ........... obstacle N = 40

Documented deviations from the reference (DESIGN.md section 4), asserted as such: for an env with a non-finite position
the shape reward and `indiv` are non-finite and nan_flag is set (scipy's directed_hausdorff skips NaN distances); the
controller returns finite actions for a NaN state (fmin / fmax clip).
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import formation_gym  # noqa: E402,F401
from formation_gym import _native as nat  # noqa: E402
from formation_gym.batched import BatchedFormationEnv  # noqa: E402
from oracle import mpe_oracle as mo  # noqa: E402
from oracle import policy_oracle as po  # noqa: E402

HD, BASIC = "formation_hd_env", "basic_formation_env"
PART, RANGE, OBST = "formation_hd_partial_env", "formation_hd_partial_range_env", "formation_hd_obs_env"
F32, F64 = torch.float32, torch.float64
WL = 100                                     # episode length: no episode ends in these tests
SIZE = {HD: 0.03, BASIC: 0.1, PART: 0.04, RANGE: 0.04, OBST: 0.1}
N_GOALS, N_OBST = 4, 3                       # obstacle scenario: goal landmarks, obstacles (make_world's)
N_LM = {PART: 5, RANGE: 4}                   # partial scenarios: landmarks (make_world's)
NUM_OBS, OBS_RANGE = 3, 0.7
INF, NAN = math.inf, math.nan


def f32(x):
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float64)


def prm_for(scen, **kw):
    return mo.WorldParams(agent_size=SIZE[scen], world_length=WL, **kw)


def make_env(scen, E, N, dtype, **kw):
    extra = {}
    if scen == BASIC:
        extra["num_landmarks"] = N
    elif scen == OBST:
        extra.update(num_landmarks=N_GOALS, num_obstacles=N_OBST)
    extra.update(kw)
    return BatchedFormationEnv(scen, E, N, episode_length=WL, dtype=dtype, auto_reset=False, seed=0, **extra)


def to_dev(x, dtype):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype, device="cuda")


def host(t):
    return t.detach().double().cpu().numpy()


def oracle_step(scen, st, act, prm):
    """One env.step of the oracle from the state dict `st` (numpy fp64) -> new state dict + outputs."""
    step = np.zeros(st["pos"].shape[0], np.int64)
    with np.errstate(all="ignore"):
        if scen == HD:
            r = mo.hd_env_step(st["pos"], st["vel"], act, st["shape"], st["ivel"], step, prm)
            nxt = dict(st, pos=r["pos"], vel=r["vel"])
        elif scen == BASIC:
            r = mo.basic_env_step(st["pos"], st["vel"], act, st["lm"], step, prm)
            nxt = dict(st, pos=r["pos"], vel=r["vel"])
        elif scen in (PART, RANGE):
            r = mo.partial_env_step(st["pos"], st["vel"], act, st["lm"], step, prm=prm,
                                    num_obs=NUM_OBS if scen == PART else None,
                                    obs_range=OBS_RANGE if scen == RANGE else None)
            nxt = dict(st, pos=r["pos"], vel=r["vel"])
        else:
            r = mo.obstacle_env_step(st["pos"], st["vel"], act, st["lm"][:, :N_GOALS], st["lm"][:, N_GOALS:],
                                     st["lmv"][:, N_GOALS:], step, prm)
            lm = np.concatenate([st["lm"][:, :N_GOALS], r["obst"]], 1)
            lmv = np.concatenate([st["lmv"][:, :N_GOALS], r["obst_vel"]], 1)
            nxt = dict(st, pos=r["pos"], vel=r["vel"], lm=lm, lmv=lmv)
    return nxt, r


def load_state(env, st):
    d = env.dtype
    env.pos.copy_(to_dev(st["pos"], d))
    env.vel.copy_(to_dev(st["vel"], d))
    if "shape" in st:
        env.ideal_shape.copy_(to_dev(st["shape"], d))
        env.ideal_vel.copy_(to_dev(st["ivel"], d))
    if "lm" in st:
        env.landmarks.copy_(to_dev(st["lm"], d))
    if "lmv" in st:
        env.landmark_vel.copy_(to_dev(st["lmv"], d))


def sub(st, idx):
    return {k: v[idx] for k, v in st.items()}


def assert_pattern(got, want, tol, what):
    """Same NaN / +inf / -inf entries; finite entries within tol."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    for f in (np.isnan, np.isposinf, np.isneginf):
        bad = f(got) != f(want)
        assert not bad.any(), "%s: %s differs at %s (got %s, want %s)" % (
            what, f.__name__, np.argwhere(bad)[:4].tolist(), got[bad][:4], want[bad][:4])
    fin = np.isfinite(want)
    if fin.any():
        err = float(np.abs(got[fin] - want[fin]).max())
        assert err <= tol, "%s: max abs err %.3e > %.1e" % (what, err, tol)


# ====================================================================== a. non-finite propagation
class Path:
    def __init__(self, pid, scen, N, dtype, span, opts=None, bfs=0, tol=None, kinds="all", **kw):
        self.id, self.scen, self.N, self.dtype, self.span = pid, scen, N, dtype, span
        self.opts, self.bfs, self.kw, self.kinds = dict(opts or {}), bfs, kw, kinds
        self.tol = tol if tol is not None else (1e-5 if dtype == F32 else 1e-12)


def _paths():
    P = []
    for N in (3, 4, 8, 9, 16, 25, 27, 32):
        P.append(Path("hd-warp-std-f32-n%d" % N, HD, N, F32, 32 // N))
        for wobs in (1, 0):
            P.append(Path("hd-warp-gen-f32-n%d-obs%d" % (N, wobs), HD, N, F32, 32 // N, dict(no_std_kernel=1),
                          write_obs=bool(wobs)))
            P.append(Path("hd-warp-f64-n%d-obs%d" % (N, wobs), HD, N, F64, 32 // N, write_obs=bool(wobs)))
    for dt, tag in ((F32, "f32"), (F64, "f64")):
        P.append(Path("basic-warp-%s-n3" % tag, BASIC, 3, dt, 10))
        P.append(Path("hd-warp-bfs3-%s-n9" % tag, HD, 9, dt, 3, bfs=3))
        P.append(Path("hd-warp-bfs2-%s-n4" % tag, HD, 4, dt, 8, bfs=2))
        P.append(Path("tile-scalar-%s-n9" % tag, HD, 9, dt, 28, dict(force_tile_kernel=1)))
        P.append(Path("tile-scalar-%s-n10" % tag, HD, 10, dt, 25))
        P.append(Path("tile-het-%s-n9" % tag, HD, 9, dt, 28, agent_mass=[1.0 + 0.25 * (i % 3) for i in range(9)]))
        P.append(Path("lm-warp-partial-%s-n4" % tag, PART, 4, dt, 8))
        P.append(Path("lm-warp-range-%s-n5" % tag, RANGE, 5, dt, 6))
        P.append(Path("lm-warp-obst-%s-n4" % tag, OBST, 4, dt, 8, tol=2e-5 if dt == F32 else 1e-11))
        P.append(Path("tile-obst-%s-n40" % tag, OBST, 40, dt, 6, tol=2e-5 if dt == F32 else 1e-11))
    P.append(Path("tile-scalar-f32-n81", HD, 81, F32, 3, dict(no_fast_pairs=1), kinds="pos"))
    P.append(Path("tile-packed-f32-n81-obs", HD, 81, F32, 3, kinds="pos"))
    for N in (40, 243):
        for cells in (1, 0):
            P.append(Path("tile-packed-f32-n%d-%s" % (N, "cells" if cells else "filters"), HD, N, F32, 256 // N,
                          dict(no_cells=1 - cells), kinds="all" if N == 40 else "pos", write_obs=False))
    return P


PATHS = _paths()


def _kinds(path):
    """(target, value) poisons, one per env; the first component of agent `i` unless noted."""
    k = [("pos", NAN), ("pos", INF), ("pos", -INF), ("pos2", INF)]
    if path.kinds == "pos":
        return k + [("act", INF)] if not path.bfs else k
    k += [("vel", NAN), ("vel", INF), ("vel", -INF)]
    if not path.bfs:                                      # the controller writes the actions itself
        k += [("act", NAN), ("act", INF), ("act", -INF)]
        if path.dtype == F64:
            k.append(("act", 1e308))                      # finite, overflows once multiplied by the sensitivity
    if path.scen == HD:
        k += [("shape", NAN), ("ivel", NAN)]
    else:
        k.append(("lm", NAN))
    if path.scen == OBST:
        k += [("obst", NAN), ("obst", INF), ("obst", -INF)]
    return k


def _state(path, E, rng):
    N, s = path.N, SIZE[path.scen]
    spread = 1.6 * s * math.sqrt(N) + s                   # dense: contacts and reward collisions occur
    st = {"pos": f32(rng.uniform(-spread, spread, (E, N, 2))), "vel": f32(rng.uniform(-0.3, 0.3, (E, N, 2)))}
    if path.scen == HD:
        lm = rng.uniform(-1, 1, (E, N, 2))
        st["shape"] = f32(lm - lm.mean(1, keepdims=True))
        st["ivel"] = f32(rng.uniform(-1, 1, (E, 2)))
    elif path.scen == BASIC:
        st["lm"] = f32(rng.uniform(-0.5, 0.5, (E, N, 2)))
    elif path.scen in (PART, RANGE):
        st["lm"] = f32(rng.uniform(-0.5, 0.5, (E, N_LM[path.scen], 2)))
    else:
        goals = rng.uniform(-1, 1, (E, N_GOALS, 2))
        obst = rng.uniform(-spread, spread, (E, N_OBST, 2))
        st["lm"] = f32(np.concatenate([goals, obst], 1))
        st["lmv"] = np.zeros((E, N_GOALS + N_OBST, 2))
        st["lmv"][:, N_GOALS:, 1] = -1.0
    return st


def _poison(st, acts, e, kind, N, rng):
    tgt, val = kind
    i, c = int(rng.integers(0, N)), int(rng.integers(0, 2))
    if tgt == "pos":
        st["pos"][e, i, c] = val
    elif tgt == "pos2":                                   # two poisoned agents in one env
        j = (i + 1 + int(rng.integers(0, N - 1))) % N
        st["pos"][e, i, 0] = val
        st["pos"][e, j, 1] = -val
    elif tgt == "vel":
        st["vel"][e, i, c] = val
    elif tgt == "act":
        acts[0][e, i, c] = val                            # only the first step's action
    elif tgt == "shape":
        st["shape"][e, i, c] = val
    elif tgt == "ivel":
        st["ivel"][e, c] = val
    elif tgt == "lm":
        st["lm"][e, i % (N_GOALS if "lmv" in st else st["lm"].shape[1]), c] = val
    elif tgt == "obst":
        st["lm"][e, N_GOALS + i % N_OBST, c] = val


KEYS = ("pos", "vel", "obs", "indiv", "reward", "done", "step_count", "ep_return", "ep_collisions", "nan_flag",
        "landmarks", "landmark_vel")


def _run(path, E, st, acts, steps=3):
    """Kernel run from `st`; per step: snapshot of every buffer and the actions the step consumed."""
    snaps = []
    with nat.options(**path.opts):
        env = make_env(path.scen, E, path.N, path.dtype, **path.kw)
        load_state(env, st)
        for t in range(steps):
            if path.bfs:
                used = (env.bfs_actions(path.bfs) if t == 0 else env.actions).clone()
                env.step_bfs(path.bfs)
            else:
                used = to_dev(acts[t], path.dtype)
                env.step(used)
            torch.cuda.synchronize()
            snap = {k: getattr(env, k).clone() for k in KEYS if getattr(env, k, None) is not None}
            snap["act"] = used
            snaps.append(snap)
    return snaps


@pytest.mark.parametrize("placement", ["first", "last"])
@pytest.mark.parametrize("path", PATHS, ids=[p.id for p in PATHS])
def test_nonfinite_state_matches_reference(path, placement):
    """One poison per env -- NaN / +-inf in one agent's position, velocity or action (1e308 in fp64), in the ideal
    shape, ideal_vel, a landmark or an obstacle, or two agents at once -- at the first or the last env slot of a warp
    span / CTA tile, plus +inf in the ragged tail (E = span * (2K + 2) + 1).  Three steps, no auto-reset, checked
    after every step against the fp64 oracle (chained on its own outputs in the fp64 build, restarted from the
    kernel's state in the fp32 build): the NaN / +-inf pattern of pos, vel, obs, landmarks and obstacles, finite
    entries to 1e-12 (fp64) / 1e-5 (fp32), nan_flag on exactly the envs with a non-finite position, and every other
    env bit-identical to a run without the poisons (nothing leaks across a warp or a CTA)."""
    if path.span == 1 and placement == "last":
        pytest.skip("one env per span: first == last")
    N, span = path.N, path.span
    kinds = _kinds(path)
    K = len(kinds)
    E = span * (2 * K + 2) + 1
    rng = np.random.default_rng(N * 131 + K + (7 if placement == "last" else 0))
    st = _state(path, E, rng)
    acts = [f32(rng.uniform(-1, 1, (E, N, 2))) for _ in range(3)]
    clean = _run(path, E, st, acts)

    pst = {k: v.copy() for k, v in st.items()}
    pacts = [a.copy() for a in acts]
    where = {}
    for k, kind in enumerate(kinds):
        e = span * (2 * k + 1) + (0 if placement == "first" else span - 1)
        _poison(pst, pacts, e, kind, N, rng)
        where[e] = kind
    _poison(pst, pacts, E - 1, ("pos", INF), N, rng)     # alone in the ragged last span
    where[E - 1] = ("pos", INF)
    got = _run(path, E, pst, pacts)

    idx = np.array(sorted(where))
    others = torch.ones(E, dtype=torch.bool, device="cuda")
    others[torch.as_tensor(idx, device="cuda")] = False
    prm = prm_for(path.scen, **({"agent_mass": path.kw["agent_mass"]} if "agent_mass" in path.kw else {}))
    ost = sub(pst, idx)
    flagged = np.zeros(len(idx), bool)
    for t in range(3):
        g, c = got[t], clean[t]
        for key in c:
            if key in ("act",):
                continue
            if key in ("done", "step_count"):
                assert torch.equal(g[key], c[key]), (t, key)
            else:
                assert torch.equal(g[key][others], c[key][others]), (t, key)
        if path.dtype == F32 and t > 0:                       # restart from the kernel's (fp32) state
            ost = dict(ost, **sub(read_state_snap(got[t - 1], ost), idx))
        act = host(g["act"])[idx]
        ost, r = oracle_step(path.scen, ost, act, prm)
        tag = "step %d" % (t + 1)
        assert_pattern(host(g["pos"])[idx], r["pos"], path.tol, tag + " pos")
        assert_pattern(host(g["vel"])[idx], r["vel"], path.tol * (10 if path.scen == OBST else 1), tag + " vel")
        if "obs" in g:
            assert_pattern(host(g["obs"])[idx], r["obs"], path.tol * (10 if path.scen == OBST else 1), tag + " obs")
        if path.scen != HD:
            assert_pattern(host(g["landmarks"])[idx], ost["lm"], path.tol, tag + " landmarks")
        if path.scen == OBST:
            assert_pattern(host(g["landmark_vel"])[idx], ost["lmv"], 0.0, tag + " obstacle velocities")
        flagged |= ~np.isfinite(r["pos"]).all(axis=(1, 2))
        assert np.array_equal(host(g["nan_flag"])[idx] != 0, flagged), tag + " nan_flag"
        indiv = host(g["indiv"])[idx]
        for q, e in enumerate(idx):
            if flagged[q] and path.scen != BASIC:             # documented: the shape term turns NaN (DESIGN.md 4)
                assert not np.isfinite(indiv[q]).any() and not np.isfinite(host(g["reward"])[e]).any(), (tag, e)
            elif where[e][0] not in ("shape", "lm") or path.scen == BASIC:   # (a NaN shape / goal: DESIGN.md 4)
                assert_pattern(indiv[q], r["indiv"][q], path.tol * 10, "%s indiv env %d %s" % (tag, e, where[e]))
    # the inf cases are what the NaN-keeping cut-off test used to drop: make sure they did reach the partners
    for q, e in enumerate(idx):
        if where[e] in (("pos", INF), ("pos", -INF), ("pos2", INF)):
            assert np.isnan(host(got[-1]["pos"])[e]).any(), e


def read_state_snap(snap, like):
    out = {"pos": host(snap["pos"]), "vel": host(snap["vel"])}
    for k, b in (("lm", "landmarks"), ("lmv", "landmark_vel")):
        if k in like:
            out[k] = host(snap[b])
    return out


# ---- the controller keeps finite actions on a NaN state (documented deviation, DESIGN.md 4)
def test_controller_on_nan_state_returns_finite_actions():
    E, N = 4, 9
    rng = np.random.default_rng(3)
    pos = f32(rng.uniform(-1, 1, (E, N, 2)))
    shape = f32(rng.uniform(-1, 1, (E, N, 2)))
    ivel = f32(rng.uniform(-1, 1, (E, 2)))
    pos[1, 4, 0] = NAN
    for dtype in (F32, F64):
        env = make_env(HD, E, N, dtype)
        load_state(env, dict(pos=pos, vel=np.zeros_like(pos), shape=shape, ivel=ivel))
        act = host(env.bfs_actions(3))
        assert np.isfinite(act).all()
        want = po.bfs_actions_batch(pos[[0, 2, 3]], shape[[0, 2, 3]], ivel[[0, 2, 3]], 3)
        assert np.abs(act[[0, 2, 3]] - want).max() <= (1e-12 if dtype == F64 else 1e-5)


# ====================================================================== b. threshold boundaries
def _ulps(x, k, dtype=np.float64):
    """x moved by k ulps of `dtype` (k may be negative)."""
    x = dtype(x)
    for _ in range(abs(k)):
        x = np.nextafter(x, dtype(INF) if k > 0 else dtype(-INF))
    return float(x)


def boundary_offsets(thr, rng, ftype=np.float64, count=16):
    """Pair offsets (dx, dy) of `ftype` whose np.linalg.norm lands on, next to or across `thr`.
    fp64: axis-aligned at thr and thr +- 1..4 ulp; directions where sqrt(fma(y, y, x*x)) (the reference's norm) and
    sqrt(x*x + y*y) fall on different sides of thr; directions where the fma form hits thr exactly.
    fp32: axis-aligned and diagonal at thr +- 1..8 fp32 ulp (the fp32 build is compared outside +-4 ulp)."""
    offs = [(float(ftype(thr)), 0.0), (0.0, -float(ftype(thr)))]
    ks = (-4, -3, -2, -1, 1, 2, 3, 4) if ftype == np.float64 else (-8, -7, -6, -5, -1, 1, 5, 6, 7, 8)
    for k in ks:
        offs.append((_ulps(thr, k, ftype), 0.0))
    if ftype == np.float32:
        u = float(np.spacing(np.float32(thr)))
        for k in (-8, -6, 6, 8):
            a = rng.uniform(0, 2 * math.pi)
            r = thr + k * u
            offs.append((float(np.float32(r * math.cos(a))), float(np.float32(r * math.sin(a)))))
        return offs
    straddle, exact = [], []
    for _ in range(200000):
        if len(straddle) >= count // 2 and len(exact) >= count // 2:
            break
        a = rng.uniform(0, 2 * math.pi)
        x, y = thr * math.cos(a), thr * math.sin(a)
        fma = float(mo.norm2(np.float64(x), np.float64(y)))
        plain = math.sqrt(x * x + y * y)
        if (fma < thr) != (plain < thr):
            if len(straddle) < count // 2:
                straddle.append((x, y))
        elif fma == thr and len(exact) < count // 2:
            exact.append((x, y))
    assert len(straddle) >= 2 and len(exact) >= 2
    return offs + straddle + exact


def _far_point(k, N):
    return (3.0 + 0.7 * k, -2.0 - 0.45 * k)


def _boundary_batch(scen, N, thr, rng, ftype=np.float64):
    """One env per offset: agent 0 at the origin, agent 1 at the offset (so p_1 - p_0 is the offset exactly), the
    others far apart."""
    offs = boundary_offsets(thr, rng, ftype)
    E = len(offs)
    pos = np.zeros((E, N, 2))
    for e, (dx, dy) in enumerate(offs):
        pos[e, 1] = (dx, dy)
        for k in range(2, N):
            pos[e, k] = _far_point(k, N)
    return pos


def _run_still(path_opts, scen, N, dtype, st, kw=None):
    kw = dict(kw or {})
    with nat.options(**path_opts):
        env = make_env(scen, st["pos"].shape[0], N, dtype, contact_force=0.0, **kw)
        load_state(env, st)
        obs, rew, done, info = env.step(torch.zeros(st["pos"].shape[0], N, 2, dtype=dtype, device="cuda"))
        torch.cuda.synchronize()
    return env


def _still_state(scen, pos, rng):
    E, N = pos.shape[:2]
    st = {"pos": pos, "vel": np.zeros_like(pos)}
    if scen == HD:
        st["shape"] = np.zeros((E, N, 2)); st["shape"][:, :, 0] = np.linspace(-0.5, 0.5, N)
        st["ivel"] = np.zeros((E, 2))
    elif scen == BASIC:
        st["lm"] = np.tile(np.linspace(-0.5, 0.5, N)[None, :, None], (E, 1, 2))
    elif scen in (PART, RANGE):
        ring = [[0.5, 0.5], [-0.5, 0.5], [0.0, -0.5], [0.5, -0.25], [-0.5, -0.25]][:N_LM[scen]]
        st["lm"] = np.tile(np.array(ring)[None], (E, 1, 1))
    else:
        goals = np.tile(np.array([[0.5, 0.5], [-0.5, 0.5], [0.0, -0.5], [0.5, -0.25]])[None], (E, 1, 1))
        obst = np.tile(np.array([[-6.0, 5.0], [-7.0, 5.0], [-8.0, 5.0]])[None], (E, 1, 1))
        st["lm"] = np.concatenate([goals, obst], 1)
        st["lmv"] = np.zeros((E, N_GOALS + N_OBST, 2))
    return st


# (scenario, N, collision threshold, kernel-path options, extra env arguments, id)
THRESHOLD_CASES = [
    (HD, 3, 0.03, {}, {}, "hd-warp-n3"),
    (HD, 9, 0.03, {}, {}, "hd-warp-n9"),
    (HD, 9, 0.03, dict(force_tile_kernel=1), {}, "hd-tile-n9"),
    (HD, 40, 0.03, {}, dict(write_obs=False), "hd-packed-n40"),
    (HD, 40, 0.03, dict(no_cells=1), dict(write_obs=False), "hd-packed-filters-n40"),
    (BASIC, 3, 0.2, {}, {}, "basic-warp-n3"),
    (BASIC, 3, 0.2, dict(force_tile_kernel=1), {}, "basic-tile-n3"),
    (PART, 4, 0.08, {}, {}, "partial-lm-warp-n4"),
    (RANGE, 5, 0.08, {}, {}, "range-lm-warp-n5"),
    (RANGE, 5, 0.08, dict(force_tile_kernel=1), {}, "range-tile-n5"),
    (OBST, 4, 0.2, {}, {}, "obst-lm-warp-n4"),
    (OBST, 40, 0.2, {}, {}, "obst-tile-n40"),
]


def _collisions_ref(scen, r_indiv, N):
    """Per-env collision total from the oracle's individual rewards: agent N-1 is far from everything, so its reward
    is the shared base term (minus its self-collision in basic_formation_env)."""
    pen = 2.0 if scen == OBST else 1.0
    base = r_indiv[:, -1:] + (1.0 if scen == BASIC else 0.0)
    return np.rint((base - r_indiv).sum(1) / pen).astype(np.int64)


def _oracle_still(scen, st, prm):
    E, N = st["pos"].shape[:2]
    _, r = oracle_step(scen, st, np.zeros((E, N, 2)), prm)
    return r


@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("scen,N,thr,opts,kw,cid", THRESHOLD_CASES, ids=[c[-1] for c in THRESHOLD_CASES])
def test_collision_threshold_boundaries(scen, N, thr, opts, kw, cid, dtype):
    """Pairs at exactly the reward's collision threshold (hd (s_i+s_j)/2, basic / partial / obstacle s_i+s_j), at
    +-1..4 ulp, and in directions where the reference's fma-contracted norm and the plain one disagree about the side.
    contact_force = 0, zero velocities and actions: the step leaves the positions where they were put.  fp64:
    individual rewards and ep_collisions equal to the oracle's; fp32: equal outside a band of +-4 fp32 ulp."""
    rng = np.random.default_rng(int(thr * 1e4) + N)
    pos = _boundary_batch(scen, N, thr, rng, np.float64 if dtype == F64 else np.float32)
    if dtype == F32:
        pos = f32(pos)
    st = _still_state(scen, pos, rng)
    prm = prm_for(scen, contact_force=0.0)
    r = _oracle_still(scen, st, prm)
    env = _run_still(opts, scen, N, dtype, st, kw)
    assert np.array_equal(host(env.pos), pos)            # the positions did not move
    got_col = env.ep_collisions.cpu().numpy().astype(np.int64)
    want_col = _collisions_ref(scen, r["indiv"], N)
    d = pos[:, 1] - pos[:, 0]
    dist = mo.norm2(d[:, 0], d[:, 1])
    if dtype == F64:
        keep = np.ones(len(dist), bool)
    else:
        band = 4 * (np.spacing(np.float32(thr)).astype(np.float64))
        keep = np.abs(dist - thr) > band
    assert keep.sum() >= 4
    assert np.array_equal(got_col[keep], want_col[keep]), (dist[keep], got_col[keep], want_col[keep])
    tol = 1e-12 if dtype == F64 else 1e-5
    assert np.abs(host(env.indiv)[keep] - r["indiv"][keep]).max() <= tol * 10
    self_hits = N if scen == BASIC else 0
    assert (want_col[keep] > self_hits).any() and (want_col[keep] == self_hits).any()


def test_boundary_constructions_straddle_in_fp64():
    """(also checked on CPU in test_oracle_edges.py) the fp64 batch really has pairs on both sides and on thr."""
    rng = np.random.default_rng(300)
    offs = boundary_offsets(0.03, rng)
    d = np.array([float(mo.norm2(np.float64(x), np.float64(y))) for x, y in offs])
    assert (d == 0.03).any() and (d < 0.03).any() and (d > 0.03).any()


@pytest.mark.parametrize("scen,N,opts,het", [(HD, 9, {}, False), (HD, 9, dict(force_tile_kernel=1), False),
                                             (PART, 4, {}, False), (HD, 9, {}, True)],
                         ids=["warp-generic", "tile", "lm-warp", "tile-het"])
def test_speed_exactly_max_speed_is_not_clamped(scen, N, opts, het):
    """core.py:271-276 clamps when speed > max_speed: a velocity whose norm equals max_speed exactly keeps its
    components (the clamp v / sp * max_speed would move some of them by an ulp).  fp64, generic instantiations."""
    rng = np.random.default_rng(17)
    vmax = 0.6
    prm0 = prm_for(scen)
    cand = []
    while len(cand) < 16:
        a = rng.uniform(0, 2 * math.pi)
        u = np.array([[[math.cos(a), math.sin(a)]]]) * vmax / (prm0.sensitivity * prm0.dt)
        _, v = mo.world_step(np.zeros((1, 1, 2)), np.zeros((1, 1, 2)), u, mo.WorldParams(collide=False))
        sp = np.sqrt(np.square(v[..., 0]) + np.square(v[..., 1]))[0, 0]
        clamped = v[0, 0] / sp * vmax
        if sp == vmax and (clamped != v[0, 0]).any():
            cand.append(u[0, 0])
    E = len(cand)
    pos = np.zeros((E, N, 2))
    for k in range(N):
        pos[:, k] = _far_point(k, N)
    act = np.zeros((E, N, 2))
    act[:, 0] = np.array(cand)
    st = _still_state(scen, pos, rng)
    if het:
        kw = dict(agent_max_speed=[vmax] * N)
        prm = prm_for(scen, agent_max_speed=[vmax] * N)
    else:
        kw = dict(max_speed=vmax)
        prm = prm_for(scen, max_speed=vmax)
    _, r = oracle_step(scen, st, act, prm)
    with nat.options(**opts):
        env = make_env(scen, E, N, F64, **kw)
        load_state(env, st)
        env.step(to_dev(act, F64))
        torch.cuda.synchronize()
    v = host(env.vel)
    assert np.array_equal(v, r["vel"])
    sp = np.sqrt(np.square(v[:, 0, 0]) + np.square(v[:, 0, 1]))
    assert (sp == vmax).all()


@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("N,opts", [(4, {}), (40, {})], ids=["lm-warp-n4", "tile-n40"])
def test_obstacle_resting_on_the_floor_stops(N, opts, dtype):
    """formation_hd_obs_env.py:85-88: an obstacle falls at (0, -1) while y > -2.2 and stops at y == -2.2 exactly."""
    E = 4
    pos = np.zeros((E, N, 2))
    for k in range(N):
        pos[:, k] = _far_point(k, N)
    st = _still_state(OBST, pos, None)
    floor = np.float64(-2.2) if dtype == F64 else np.float64(np.float32(-2.2))
    ys = [floor, _ulps(floor, 1, np.float64 if dtype == F64 else np.float32),
          _ulps(floor, -1, np.float64 if dtype == F64 else np.float32), floor]
    for e, y in enumerate(ys):
        st["lm"][e, N_GOALS:, 1] = y
    env = _run_still(opts, OBST, N, dtype, st)
    lmv = host(env.landmark_vel)[:, N_GOALS:]
    assert np.array_equal(host(env.landmarks)[:, N_GOALS:, 1], np.array(ys)[:, None].repeat(N_OBST, 1))
    want = np.where(np.array(ys) > -2.2 if dtype == F64 else np.array(ys) > np.float32(-2.2), -1.0, 0.0)
    assert np.array_equal(lmv[:, :, 1], want[:, None].repeat(N_OBST, 1))
    assert (lmv[:, :, 0] == 0).all()


CONTACT_CASES = [
    (HD, 3, F64, {}, {}), (HD, 9, F32, {}, {}), (HD, 9, F32, dict(no_std_kernel=1), {}),
    (HD, 9, F64, dict(force_tile_kernel=1), {}), (HD, 40, F32, {}, dict(write_obs=False)),
    (HD, 40, F32, dict(no_cells=1), dict(write_obs=False)), (PART, 4, F64, {}, {}), (OBST, 40, F64, {}, {}),
]


@pytest.mark.parametrize("scen,N,dtype,opts,kw", CONTACT_CASES,
                         ids=["hd-warp-f64-n3", "hd-warp-std-f32-n9", "hd-warp-gen-f32-n9", "hd-tile-f64-n9",
                              "hd-packed-f32-n40", "hd-filters-f32-n40", "partial-lm-warp-f64-n4", "obst-tile-f64-n40"])
def test_contact_force_at_dmin_and_at_the_cutoff(scen, N, dtype, opts, kw):
    """Default contact force, pairs at d_min = 2 s and at the kernels' cut-off d_min + kcut * k (kcut = 20 in fp32,
    50 in fp64), each +-1..3 ulp: the step equals the oracle (no cut-off) to 1e-12 (fp64) / 1e-5 (fp32), which pins
    the cut-off error DESIGN.md claims."""
    s, k = SIZE[scen], 1e-3
    kcut = 50.0 if dtype == F64 else 20.0
    dmin = 2 * s
    dists = []
    for d in (dmin, dmin + kcut * k):
        for u in (-3, -2, -1, 0, 1, 2, 3):
            dists.append(_ulps(d, u, np.float64 if dtype == F64 else np.float32))
    E = len(dists)
    pos = np.zeros((E, N, 2))
    for e, d in enumerate(dists):
        pos[e, 1] = (d, 0.0) if e % 2 == 0 else (0.0, -d)           # agent 0 at the origin: p_1 - p_0 is exact
        for q in range(2, N):
            pos[e, q] = _far_point(q, N)
    if dtype == F32:
        pos = f32(pos)
    rng = np.random.default_rng(5)
    st = _still_state(scen, pos, rng)
    prm = prm_for(scen)
    _, r = oracle_step(scen, st, np.zeros((E, N, 2)), prm)
    with nat.options(**opts):
        env = make_env(scen, E, N, dtype, **kw)
        load_state(env, st)
        env.step(torch.zeros(E, N, 2, dtype=dtype, device="cuda"))
        torch.cuda.synchronize()
    tol = 1e-12 if dtype == F64 else 1e-5
    assert_pattern(host(env.pos), r["pos"], tol, "pos")
    assert_pattern(host(env.vel), r["vel"], tol, "vel")
    assert np.abs(r["vel"][:7, 0]).max() > 1e-3            # the pairs at d_min do push


# ====================================================================== c. controller ties
def _lattice_batch(E, N, rng, half=4):
    """Distinct positions and shape points on the lattice 2^-4 Z^2 in [-half/16, half/16]^2 -- in every second env
    mirror-symmetric (x -> -x), so that many distances tie exactly; ideal_vel on the same lattice."""
    grid = np.array([(x, y) for x in range(-half, half + 1) for y in range(-half, half + 1)], np.float64) / 16.0
    right = grid[grid[:, 0] > 0]
    axis = grid[grid[:, 0] == 0]

    def points(sym):
        if not sym:
            return grid[rng.choice(len(grid), N, replace=False)]
        h = right[rng.choice(len(right), N // 2, replace=False)]
        mid = axis[rng.choice(len(axis), N % 2, replace=False)]
        return np.concatenate([h, h * np.array([-1.0, 1.0]), mid])

    pos = np.stack([points(e % 2 == 1) for e in range(E)])
    shape = np.stack([points(e % 2 == 1) for e in range(E)])
    ivel = rng.integers(-16, 17, (E, 2)) / 16.0
    return pos, shape, ivel


# fp32 only at power-of-two fan-outs: at n = 3 the group means are inexact and a tie breaks by rounding
BFS_TIES = [(9, 3, F64), (16, 4, F64), (8, 2, F64), (64, 8, F64), (16, 4, F32), (8, 2, F32), (64, 8, F32)]


@pytest.mark.parametrize("N,n,dtype", BFS_TIES, ids=["n%d-fan%d-%s" % (c[0], c[1], "f64" if c[2] == F64 else "f32")
                                                      for c in BFS_TIES])
def test_controller_ties_on_a_dyadic_lattice(N, n, dtype):
    """get_action_BFS on lattice states with exact distance ties, against the oracle's stable argsort (np.argmin
    takes the first minimum).  fp64 to 1e-12; fp32 at power-of-two fan-outs, where the distances and group means the
    controller compares are exact on these inputs, to 1e-5 on every sample -- no sample may take the other branch."""
    rng = np.random.default_rng(N * 10 + n)
    E = 256 if N <= 16 else 64
    pos, shape, ivel = _lattice_batch(E, N, rng, half=8 if N == 64 else 4)
    want = po.bfs_actions_batch(pos, shape, ivel, n)
    env = make_env(HD, E, N, dtype)
    load_state(env, dict(pos=pos, vel=np.zeros_like(pos), shape=shape, ivel=ivel))
    got = host(env.bfs_actions(n))
    err = np.abs(got - want).max(axis=(1, 2))
    assert err.max() <= (1e-12 if dtype == F64 else 1e-5), (np.flatnonzero(err > 1e-12), err.max())


STEP_TIES = [(4, 2), (8, 2), (16, 4)]


@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("N,n", STEP_TIES, ids=["n%d-fan%d" % c for c in STEP_TIES])
def test_step_bfs_ties_on_a_dyadic_lattice(N, n, dtype):
    """The controller fused into the step kernel (step_bfs): the actions it leaves for the next step, computed from
    the new state, against the oracle's controller on the kernel's new state; the physics against the oracle."""
    rng = np.random.default_rng(N * 13 + n)
    E = 128
    pos, shape, ivel = _lattice_batch(E, N, rng, half=6)
    st = dict(pos=pos * 4, vel=np.zeros_like(pos), shape=shape, ivel=ivel)   # 1/4 apart: no contacts on the lattice
    env = make_env(HD, E, N, dtype)
    load_state(env, st)
    a0 = host(env.bfs_actions(n))
    want0 = po.bfs_actions_batch(st["pos"], shape, ivel, n)
    tol = 1e-12 if dtype == F64 else 1e-5
    assert np.abs(a0 - want0).max() <= tol
    env.step_bfs(n)
    torch.cuda.synchronize()
    _, r = oracle_step(HD, st, a0, prm_for(HD))
    assert np.abs(host(env.pos) - r["pos"]).max() <= tol
    newpos = host(env.pos)
    want1 = po.bfs_actions_batch(newpos, shape, ivel, n)
    err = np.abs(host(env.actions) - want1).max(axis=(1, 2))
    if dtype == F64:
        assert err.max() <= 1e-12
    else:                                                  # off the lattice: fp32 may take the other branch
        assert (err > 1e-5).mean() <= 0.05, err.max()
