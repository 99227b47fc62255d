"""CPU-only tests (no GPU, no compute calls into the CUDA library):
  * the C-ABI shared library loads and exports every symbol include/formation_gym_b200.h declares,
    and the ctypes mirror of its structs has the C compiler's layout;
  * host logic of the drop-in facade: make_env signature, spaces, types (API contract frozen from
    the unmodified reference in tests/golden/api_contract.json), loud failure without a device;
  * the per-object loop port used as the timed CPU baseline agrees with the golden fixtures;
  * multi-GPU plumbing on the gloo backend at world_size 2 (env-range sharding + stats all-reduce).
"""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden")
HEADER = os.path.join(ROOT, "include", "formation_gym_b200.h")


# ------------------------------------------------------------------ C ABI
def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fg_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from formation_gym import _build, _native
    _build.build()                                  # nvcc cross-compiles without a GPU
    lib = C.CDLL(_native.lib_path())
    syms = _declared_symbols()
    assert len(syms) >= 14 and "fg_step_fused" in syms and "fg_step_fused_f64" in syms
    for s in syms:
        assert hasattr(lib, s), "missing export %s" % s
    assert sorted(_native.EXPORTS) == syms          # the binding covers exactly the header
    assert _native.load().fg_abi_version() == _native.FG_ABI_VERSION == 9


def test_ctypes_structs_match_c_layout():
    """Compile a 10-line C program against the header and compare sizeof/offsetof with ctypes."""
    from formation_gym import _native
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "formation_gym_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(fg_params), sizeof(fg_buffers), sizeof(fg_wall),
         offsetof(fg_params, has_accel), offsetof(fg_params, agent_mass), offsetof(fg_params, walls),
         offsetof(fg_buffers, step), offsetof(fg_buffers, tick_dev));
  printf("%zu\n", offsetof(fg_buffers, nan_flag));
  return 0; }
'''
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "l.c"), os.path.join(d, "l")
        open(src, "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    P, B = _native.fg_params, _native.fg_buffers
    want = [C.sizeof(P), C.sizeof(B), C.sizeof(_native.fg_wall), P.has_accel.offset, P.agent_mass.offset,
            P.walls.offset, B.step.offset, B.tick_dev.offset, B.nan_flag.offset]
    assert got == want


def test_option_switches_are_validated_and_restored():
    """fg_set_option / fg_get_option (A/B switches read once, never on the launch path): unknown names and
    out-of-range values are argument errors; the context manager restores the previous values."""
    from formation_gym import _native as nat
    lib = nat.load()
    assert nat.get_option("force_tile_kernel") == 0 and nat.get_option("waves") == 1 and nat.get_option("row_nbuf") == 2
    with nat.options(force_tile_kernel=1, waves=3):
        assert nat.get_option("force_tile_kernel") == 1 and nat.get_option("waves") == 3
    assert nat.get_option("force_tile_kernel") == 0 and nat.get_option("waves") == 1
    assert lib.fg_set_option(b"waves", 0) == -1 and b"out of range" in lib.fg_last_error()
    assert lib.fg_set_option(b"no_such_switch", 1) == -1 and b"unknown option" in lib.fg_last_error()
    assert lib.fg_set_option(None, 1) == -1
    assert nat.get_option("waves") == 1


def test_bad_arguments_are_rejected_without_a_device():
    """Argument validation happens before any CUDA call: status < 0 and a message, no exception."""
    from formation_gym import _native as nat
    lib = nat.load()
    p, b = nat.make_params(), nat.fg_buffers()
    rc = lib.fg_step_fused(C.byref(p), C.byref(b), nat.FG_SCENARIO_HD, 4, 2, 2, 1, 0, 0, 0, 0, 0, None)
    assert rc == -1 and b"N >= 3" in lib.fg_last_error()
    rc = lib.fg_step_fused(C.byref(p), C.byref(b), nat.FG_SCENARIO_HD, 4, 300, 300, 1, 0, 0, 0, 0, 0, None)
    assert rc == -1 and b"FG_MAX_AGENTS" in lib.fg_last_error()
    rc = lib.fg_step_fused(C.byref(p), C.byref(b), nat.FG_SCENARIO_HD, 4, 9, 9, 1, 0, 0, 0, 0, 0, None)
    assert rc == -1 and b"non-null" in lib.fg_last_error()
    rc = lib.fg_reset(None, None, 0, 1, 3, 3, None, 0, 0, 0, None)
    assert rc == -1
    epc, thr = nat.launch_geometry(243)
    assert (epc, thr) == (1, 256)
    with pytest.raises(nat.NativeError):
        nat.ptr(__import__("torch").zeros(3))       # CPU tensors are refused: no CPU path


# ------------------------------------------------------------------ facade host logic
@pytest.mark.parametrize("scenario,n", [("formation_hd_env", 9), ("basic_formation_env", 3)])
def test_api_contract_static(scenario, n):
    import formation_gym
    from formation_gym import _native as nat
    want = json.load(open(os.path.join(GOLD, "api_contract.json")))["api"][scenario]
    np.random.seed(0)
    env = formation_gym.make_env(scenario, False, n)
    assert env.num_agents == want["num_agents"] == len(env.agents)
    assert len(env.world.landmarks) == want["n_landmarks"]
    assert env.world_length == want["world_length"]
    assert env.shared_reward == want["shared_reward"]
    assert env.world.dim_c == want["dim_c"]
    assert abs(env.world.agents[0].size - want["agent_size"]) < 1e-12
    assert list(env.observation_space[0].shape) == want["obs_space_shape"]
    assert list(env.share_observation_space[0].shape) == want["share_obs_space_shape"]
    assert list(env.action_space[0].shape) == want["action_shape"]
    assert float(env.action_space[0].low[0]) == want["action_low"]
    assert float(env.action_space[0].high[0]) == want["action_high"]
    a = env.action_space[0].sample()
    assert a.shape == (2,) and a.dtype == np.float32 and np.all(np.abs(a) <= 1)
    # README's 4-argument form (README.md:61)
    env4 = formation_gym.make_env(scenario, False, n, 25)
    assert env4.world_length == 25
    # reset_world ran on the host RNG like the reference: agents in [-1, 1]^2, zero velocity
    for ag in env.world.agents:
        assert np.all(np.abs(ag.state.p_pos) <= 1) and np.all(ag.state.p_vel == 0)
    # the step path has no CPU fallback: without a CUDA device it must fail loudly
    import torch
    if not torch.cuda.is_available():
        with pytest.raises((nat.NativeError, RuntimeError)):
            env.step([np.zeros(2) for _ in range(n)])


@pytest.mark.parametrize("scenario,n", [("formation_hd_env", 9), ("basic_formation_env", 3),
                                        ("formation_hd_partial_env", 5), ("formation_hd_partial_range_env", 4),
                                        ("formation_hd_obs_env", 4)])
def test_every_stock_scenario_is_native(scenario, n):
    """All five stock scenarios resolve to their own FG_SCENARIO_* id -- formation_hd_partial_range_env subclasses the
    partial scenario and overrides its hooks, which a plain isinstance() walk mistook for a user override (round-1
    advice) -- so construction needs no device call and env.step takes the single fused launch.  A user subclass
    that overrides a hook must get the callback path."""
    import formation_gym
    from formation_gym import _native as nat
    from formation_gym.batched import SCENARIOS
    env = formation_gym.make_env(scenario, False, n)
    sc = env._native_scenario()
    assert sc is not None and sc.native_kind == SCENARIOS[scenario]
    assert sc.native_kind == {"formation_hd_env": nat.FG_SCENARIO_HD, "basic_formation_env": nat.FG_SCENARIO_BASIC,
                              "formation_hd_partial_env": nat.FG_SCENARIO_HD_PARTIAL,
                              "formation_hd_partial_range_env": nat.FG_SCENARIO_HD_PARTIAL_RANGE,
                              "formation_hd_obs_env": nat.FG_SCENARIO_HD_OBSTACLE}[scenario]

    class Custom(type(sc)):
        def reward(self, agent, world):
            return 0.0
    c = Custom()
    from formation_gym.environment import MultiAgentEnv
    env2 = MultiAgentEnv.__new__(MultiAgentEnv)
    env2.observation_callback, env2.reward_callback = c.observation, c.reward
    assert env2._native_scenario() is None


def test_bfs_observation_consistency_check():
    """get_action_BFS(ezpolicy, ...) may only collapse to the one-launch device tree when the N observations show one
    consistent state; the fixture holds a consistent and a perturbed set made with the unmodified reference."""
    import formation_gym
    g = np.load(os.path.join(GOLD, "bfs_inconsistent_n9.npz"))
    assert formation_gym._consistent_observations(list(g["obs_clean"]), 9)
    assert not formation_gym._consistent_observations(list(g["obs_noisy"]), 9)
    bad = g["obs_clean"].copy(); bad[5, -1] += 1e-3                      # another ideal_vel in one agent's row
    assert not formation_gym._consistent_observations(list(bad), 9)
    nan = g["obs_clean"].copy(); nan[2, 7] = np.nan
    assert not formation_gym._consistent_observations(list(nan), 9)
    assert not formation_gym._consistent_observations(list(g["obs_clean"][:, :-1]), 9)


def test_make_env_rejects_unknown_scenarios_and_small_hd():
    import formation_gym
    with pytest.raises(ValueError):
        formation_gym.make_env("simple_spread", False, 9)
    env = formation_gym.make_env("formation_hd_obs_env", False, 4)      # host construction needs no device
    assert len(env.world.landmarks) == 7 and env.observation_space[0].shape == (2 + 2 * 7 + 4 * 3,)
    assert [l.movable and l.collide for l in env.world.landmarks] == [False] * 4 + [True] * 3
    with pytest.raises(Exception):
        formation_gym.make_env("formation_hd_env", False, 2)      # formation_hd_env.py:58 needs N >= 3


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gym-formation_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, os.path.join(dp, f)


# ------------------------------------------------------------------ CPU-baseline port vs golden
def _port_from_state(scenario, pos, vel, extra, world_length):
    from oracle import ref_loop_port as rp
    n = pos.shape[0]
    np.random.seed(0)
    env = rp.RefLoopEnv(scenario, n, world_length, num_landmarks=(extra["lm"].shape[0] if "lm" in extra else 3))
    for a, p, v in zip(env.agents, pos, vel):
        a.pos, a.vel = p.copy(), v.copy()
    if scenario == "formation_hd_env":
        env.ideal_shape, env.ideal_vel = extra["shape"].copy(), extra["ivel"].copy()
        for l, p in zip(env.landmarks, extra["lm"]):
            l.pos = p.copy()
    else:
        for l, p in zip(env.landmarks, extra["lm"]):
            l.pos = p.copy()
    return env


@pytest.mark.parametrize("name", ["hd_n9_clustered.npz", "hd_n3_spread.npz", "hd_n27_clustered.npz"])
def test_loop_port_matches_golden_hd(name):
    g = dict(np.load(os.path.join(GOLD, name)))
    for e in range(min(4, g["pos0"].shape[0])):
        env = _port_from_state("formation_hd_env", g["pos0"][e], g["vel0"][e],
                               dict(shape=g["shape"][e], ivel=g["ivel"][e], lm=g["lm0"][e]), 25)
        env.current_step = int(g["step0"][e])
        obs_n, rew_n, done_n, info_n = env.step(list(g["act"][e]))
        P = np.stack([a.pos for a in env.agents]); V = np.stack([a.vel for a in env.agents])
        assert np.abs(P - g["pos"][e]).max() <= 1e-12 and np.abs(V - g["vel"][e]).max() <= 1e-12
        rows = g["obs_rows"] if "obs_rows" in g else np.arange(P.shape[0])
        assert np.abs(np.stack(obs_n)[rows] - g["obs"][e]).max() <= 1e-12
        ind = np.array([i["individual_reward"] for i in info_n])
        assert np.abs(ind - g["indiv"][e]).max() <= 1e-10
        assert abs(rew_n[0][0] - g["reward"][e][0]) <= 1e-9
        assert rew_n[0] is rew_n[-1]                    # [[R]] * N aliases one list (environment.py:138)
        assert list(done_n) == list(g["done"][e])


def test_loop_port_matches_golden_basic():
    g = dict(np.load(os.path.join(GOLD, "basic_n3_clustered.npz")))
    for e in range(min(4, g["pos0"].shape[0])):
        env = _port_from_state("basic_formation_env", g["pos0"][e], g["vel0"][e], dict(lm=g["lm0"][e]), 25)
        env.current_step = int(g["step0"][e])
        obs_n, rew_n, done_n, info_n = env.step(list(g["act"][e]))
        P = np.stack([a.pos for a in env.agents])
        assert np.abs(P - g["pos"][e]).max() <= 1e-12
        assert np.abs(np.stack(obs_n) - g["obs"][e]).max() <= 1e-12
        ind = np.array([i["individual_reward"] for i in info_n])
        assert np.abs(ind - g["indiv"][e]).max() <= 1e-10


# ------------------------------------------------------------------ multi-process plumbing (gloo)
def test_shard_range_partitions_exactly():
    from formation_gym.distributed import shard_range
    for total in (0, 1, 7, 8, 1000003, 1 << 20):
        for world in (1, 2, 3, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


_GLOO_WORKER = r'''
import os, sys, json
sys.path.insert(0, os.path.join(%(root)r, "gym-formation_b200"))
import torch, torch.distributed as dist
from formation_gym import distributed as fgd
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
lo, hi = fgd.shard_range(1001, rank, world)
# per-rank statistics as the step kernels would leave them: [episodes, sum R, sum R^2, sum collisions]
R = torch.arange(lo, hi, dtype=torch.float64) * 0.5 - 100.0
stats = torch.stack([torch.tensor(float(hi - lo), dtype=torch.float64), R.sum(), (R * R).sum(),
                     torch.tensor(float(3 * (hi - lo)), dtype=torch.float64)])
out = fgd.all_reduce_stats(stats.clone())
if rank == 0:
    print(json.dumps({"lo_hi": [lo, hi], "stats": out.tolist(), "summary": fgd.summarize(out)}))
dist.destroy_process_group()
'''


def test_gloo_world_size_2_stats_allreduce():
    """One process per rank over gloo: contiguous env ranges, all-reduced statistics equal the
    single-process sums (the only collective of the design; NCCL does the same on GPUs)."""
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    with tempfile.TemporaryDirectory() as d:
        script = os.path.join(d, "w.py")
        open(script, "w").write(_GLOO_WORKER % {"root": ROOT})
        procs = []
        for r in range(2):
            env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
            procs.append(subprocess.Popen([sys.executable, script], env=env, stdout=subprocess.PIPE,
                                          stderr=subprocess.PIPE, text=True))
        outs = [p.communicate(timeout=180) for p in procs]
        for p, (o, e) in zip(procs, outs):
            assert p.returncode == 0, e[-2000:]
    res = json.loads(outs[0][0].strip().splitlines()[-1])
    R = np.arange(1001, dtype=np.float64) * 0.5 - 100.0
    assert res["lo_hi"] == [0, 501]
    assert res["stats"][0] == 1001 and res["stats"][3] == 3003
    assert abs(res["stats"][1] - R.sum()) < 1e-6 and abs(res["stats"][2] - (R * R).sum()) < 1e-3
    assert abs(res["summary"]["return_mean"] - R.mean()) < 1e-9
    assert abs(res["summary"]["return_std"] - R.std()) < 1e-6


def test_render_bridge_rgb_array_on_host():
    """env.render(mode='rgb_array') (environment.py:243-393) through the numpy rasteriser: no display, no device."""
    import formation_gym
    from formation_gym import render_bridge as rb
    from formation_gym.core import Wall
    np.random.seed(3)
    env = formation_gym.make_env("formation_hd_obs_env", False, 4)
    env.world.walls.append(Wall(orient='V', axis_pos=1.5, endpoints=(-1, 1), width=0.2))
    for k, a in enumerate(env.world.agents):
        a.state.p_pos = np.array([0.5 * k - 0.75, 0.0])
    frames = env.render(mode='rgb_array')
    assert len(frames) == 1 and frames[0].shape == (700, 700, 3) and frames[0].dtype == np.uint8
    f = frames[0].astype(int)
    assert (f[0, 0] == 255).all()                                   # background
    # camera centred on the agents' centroid (0, 0): agent 1 at (-0.25, 0) -> pixel (350 - 0.25 * 175, 350)
    px = f[350, int(350 - 0.25 * 175)]
    want = 0.5 * 255 + 0.5 * 255 * np.array([0.65, 0.65, 0.85])     # half-transparent agent colour on white
    assert np.abs(px - want).max() <= 2
    assert (f[350, int(350 + 1.5 * 175)] == 0).all()                # the wall, black
    # circle radius in pixels = size * 700 / 4
    img = rb.rasterize([(0.0, 0.0, 0.4, (1.0, 0.0, 0.0), 1.0)])
    red = (img[..., 0] == 255) & (img[..., 1] == 0)
    assert abs(red.sum() - np.pi * (0.4 * 175) ** 2) < 0.02 * np.pi * (0.4 * 175) ** 2
    assert env.render(close=True) == []


_STAND_IN_REFERENCE = {
    # a minimal package with the reference's layout and make_env / step API, so that staging and the harness are
    # exercised without a checkout of the reference
    "formation_gym/__init__.py": "def make_env(scenario_name, benchmark=False, num_agents=3):\n"
                                 "    from formation_gym.environment import MultiAgentEnv\n"
                                 "    return MultiAgentEnv(num_agents)\n",
    "formation_gym/core.py": "class World(object):\n    world_length = 25\n",
    "formation_gym/environment.py": "from formation_gym.core import World\n\n\n"
                                    "class MultiAgentEnv(object):\n"
                                    "    def __init__(self, n):\n"
                                    "        self.n, self.world, self.t = n, World(), 0\n\n"
                                    "    def reset(self):\n"
                                    "        self.t = 0\n"
                                    "        return [[0.0]] * self.n\n\n"
                                    "    def step(self, act_n):\n"
                                    "        self.t += 1\n"
                                    "        done = self.t >= self.world.world_length\n"
                                    "        return [[0.0]] * self.n, [[0.0]] * self.n, [done] * self.n, [{}] * self.n\n",
    "formation_gym/scenario.py": "class BaseScenario(object):\n    pass\n",
    "formation_gym/envs/__init__.py": "",
    "formation_gym/envs/formation_hd_env.py": "from formation_gym.scenario import BaseScenario\n\n\n"
                                              "class Scenario(BaseScenario):\n    pass\n",
}


def test_staged_reference_is_byte_identical_and_runs():
    """oracle/make_ref.py stages the files of the reference's step path byte for byte (sha256 manifest) into a
    git-ignored directory like oracle/_ref, and the harness runs an env from that copy.  The source is a stand-in
    tree with the reference's layout."""
    import hashlib
    from oracle import make_ref
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "reference")
        for rel, text in _STAND_IN_REFERENCE.items():
            os.makedirs(os.path.dirname(os.path.join(src, rel)), exist_ok=True)
            open(os.path.join(src, rel), "w").write(text)
        dst = make_ref.make(src=src, dst=os.path.join(d, "_ref"), quiet=True)
        assert make_ref.staged_ok(dst)
        man = json.load(open(os.path.join(dst, "MANIFEST.json")))["files"]
        assert "formation_gym/core.py" in man and "formation_gym/envs/formation_hd_env.py" in man
        assert sorted(man) == sorted(_STAND_IN_REFERENCE)
        for rel, h in man.items():
            assert hashlib.sha256(open(os.path.join(src, rel), "rb").read()).hexdigest() == h
        env = dict(os.environ, FG_REFERENCE_ROOT=dst)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_harness.py"), "--agents", "3", "--procs", "1",
                              "--max-steps", "5", "--warmup", "1"], capture_output=True, text=True, timeout=300, env=env)
        r = json.loads(out.stdout.strip().splitlines()[-1])
        assert r["env_steps"] == 5 and r["reference_root"] == dst
        open(os.path.join(dst, "formation_gym", "core.py"), "a").write("\n# tampered\n")
        assert not make_ref.staged_ok(dst)


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` (the reference's per-env CPU loop on the host cores) needs no GPU and prints exactly
    one JSON line with the contract's keys."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "agent-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 3 and d["gpu_launches"] == 0
    # the CPU arm is the UNMODIFIED reference whenever a tree is available (/root/reference here, oracle/_ref on the
    # GPU box); the loop port is only the fallback
    from oracle import make_ref
    have = os.path.isfile("/root/reference/formation_gym/core.py") or make_ref.staged_ok()
    assert d["cpu_baseline"]["kind"] == ("reference" if have else "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["scenario"] == "formation_hd_env" and d["config"]["agents"] == 9
