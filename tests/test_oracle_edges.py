"""CPU checks of the edge-state constructions of test_gpu_edges.py and of the reference arithmetic they rely on."""
import math

import numpy as np
import pytest

from oracle import mpe_oracle as mo
from oracle import policy_oracle as po
from test_gpu_edges import BASIC, HD, OBST, PART, boundary_offsets, _boundary_batch, _lattice_batch, _still_state, \
    _collisions_ref, oracle_step, prm_for


@pytest.mark.parametrize("thr", [0.03, 0.2, 0.08, 0.25])
def test_boundary_offsets_hit_and_straddle_the_threshold(thr):
    """fp64 constructions: some pairs exactly on thr in the reference's norm, some on either side, and directions
    where the fma-contracted norm and the plain sqrt(x*x + y*y) decide differently."""
    offs = boundary_offsets(thr, np.random.default_rng(int(thr * 1e4)))
    d = np.array([float(mo.norm2(np.float64(x), np.float64(y))) for x, y in offs])
    plain = np.array([math.sqrt(x * x + y * y) for x, y in offs])
    assert (d == thr).sum() >= 3 and (d < thr).any() and (d > thr).any()
    assert ((d < thr) != (plain < thr)).sum() >= 2
    # the +-k ulp axis-aligned pairs sit k ulp away, in order
    axis = d[2:10]
    assert np.all(np.diff(axis) > 0) and axis[3] < thr < axis[4]


@pytest.mark.parametrize("thr", [0.03, 0.2, 0.08, 0.25])
def test_fp32_boundary_offsets_leave_the_band(thr):
    """fp32 constructions: besides the pairs inside +-4 fp32 ulp of thr, at least eight pairs 5..8 ulp away, on both
    sides -- the ones the fp32 build must decide like the reference."""
    offs = boundary_offsets(thr, np.random.default_rng(1), np.float32)
    d = np.array([float(mo.norm2(np.float64(x), np.float64(y))) for x, y in offs])
    band = 4 * float(np.spacing(np.float32(thr)))
    out = np.abs(d - thr) > band
    assert out.sum() >= 8 and (d[out] < thr).any() and (d[out] > thr).any()


@pytest.mark.parametrize("scen,N,thr", [(HD, 3, 0.03), (HD, 40, 0.03), (BASIC, 3, 0.2), (PART, 4, 0.08),
                                        (OBST, 4, 0.2)])
def test_boundary_batches_collide_exactly_as_placed(scen, N, thr):
    """In the oracle (contact force 0, still agents) agents 0 and 1 collide iff their norm is below thr, and the
    count the GPU test reads back from the individual rewards is that."""
    rng = np.random.default_rng(3)
    pos = _boundary_batch(scen, N, thr, rng)
    st = _still_state(scen, pos, rng)
    _, r = oracle_step(scen, st, np.zeros_like(pos), prm_for(scen, contact_force=0.0))
    assert np.array_equal(r["pos"], pos)
    d = pos[:, 1] - pos[:, 0]
    hit = mo.norm2(d[:, 0], d[:, 1]) < thr
    want = 2 * hit.astype(np.int64) + (N if scen == BASIC else 0)
    assert np.array_equal(_collisions_ref(scen, r["indiv"], N), want)
    assert hit.any() and (~hit).any()


def test_reference_contact_force_of_an_infinite_pair_is_nan():
    """core.py:304-312 with one agent at +-inf: dist = inf, pen = logaddexp(0, -inf) * k = 0, so
    force = contact_force * delta / dist * pen is NaN in the infinite component -- the pair must reach the contact
    force, as it does in the reference.  One step later the NaN has reached every partner."""
    for val in (math.inf, -math.inf):
        pos = np.array([[[0.0, 0.0], [0.5, 0.0], [val, 0.2]]])
        act = np.zeros_like(pos)
        with np.errstate(all="ignore"):
            p1, v1 = mo.world_step(pos, np.zeros_like(pos), act)
            assert np.isnan(v1[0, :, 0]).all() and np.isfinite(v1[0, :, 1]).all()
            delta = pos[0, 0] - pos[0, 2]
            dist = mo.norm2(delta[0], delta[1])
            pen = np.logaddexp(0, -(dist - 0.06) / 1e-3) * 1e-3
            assert math.isinf(dist) and pen == 0.0 and np.isnan(100.0 * delta[0] / dist * pen)
    # the issue's two-step example: the infinite position comes from an action, the NaN follows a step later
    pos = np.array([[[0.0, 0.0], [0.5, 0.0], [1.0, 0.2]]])
    act = np.array([[[0.0, 0.0], [0.0, 0.0], [math.inf, 0.0]]])
    with np.errstate(all="ignore"):
        p1, v1 = mo.world_step(pos, np.zeros_like(pos), act)
        assert np.isinf(p1[0, 2, 0]) and np.isfinite(p1[0, :2]).all()
        p2, _ = mo.world_step(p1, v1, np.zeros_like(act))
    assert np.isnan(p2[0, :, 0]).all()


def test_lattice_states_hold_exact_ties():
    """The controller-tie batches are fp32-exact, hold distinct agents and exact distance ties; the group means the
    controller sorts by are exact at a power-of-two fan-out, so the fp32 build has no excuse to take another branch."""
    rng = np.random.default_rng(8)
    pos, shape, ivel = _lattice_batch(32, 8, rng)
    assert np.array_equal(pos, np.float32(pos)) and np.array_equal(shape, np.float32(shape))
    ties = 0
    for e in range(pos.shape[0]):
        d = np.sort([float(np.hypot(*(shape[e, a] - pos[e, 0]))) for a in range(8)])
        ties += int((np.diff(d) == 0).any())
        assert len({tuple(p) for p in pos[e]}) == 8
    assert ties >= 8
    means = pos.reshape(32, 2, 4, 2).mean(2)
    assert np.array_equal(means, np.float32(means)) and np.array_equal(means * 64, np.rint(means * 64))
    assert np.isfinite(po.bfs_actions_batch(pos, shape, ivel, 2)).all()
