"""cfg3-class fixture (Hide&Seek-class arena: 49 bodies, 6 agents, wedge and
hexagonal-prism hulls, doors latched by fixed joints to static walls, grab =
fixed joint, shove = one-step hinge joint, episode resets that destroy and
recreate 27 bodies and every joint): B200 engine vs the reference CPU backend.

BIT-EXACT on every exported column: entity IDs (gen + id), row order of the
dynamic body table, joint counts, done flags and every float (positions,
rotations, velocities, rewards, lidar depths, line-of-sight flags).  Covers
src/physics/xpbd.cpp:607-718 incl. the Hinge branch (:686), narrowphase hulls
with more than 6 faces / non-quad faces, > 4-point manifolds
(narrowphase.cpp:771-879)."""
import os

import numpy as np
import pytest

from oracle import runner
from sims import SIMS
from trace_utils import assert_matches_digest_golden, assert_traces_equal, load_golden, make_inputs, rollout_gpu

EXACT = os.environ.get("MADRONA_B200_FAST_MATH", "0") != "1"
CFG = {"episode_len": 90, "seed": 17}
BODIES = 42          # PhysicsEntity rows per world (49 bodies - 6 agents - ... see sim.hpp)


@pytest.mark.skipif(not runner.available("arena"), reason="oracle/_ref not built")
def test_reference_backend_reproduces_golden():
    W, steps, ins, outs = load_golden("arena_w2_s200")
    got, _ = runner.run_reference(SIMS["arena"], W, steps, ins, CFG, workers=1)
    assert_traces_equal(got, outs)


def test_golden_exercises_joints_and_churn():
    W, steps, ins, outs = load_golden("arena_w2_s200")
    pos = outs["body_pos"]
    assert all(len(f) == BODIES * W for f in pos)
    allp = np.concatenate(pos)
    assert np.isfinite(allp).all() and allp[:, 2].min() > -0.05
    jc = outs["joint_count"][..., 0]
    # two latches at the start of every episode, unlatching and grabs / shoves change the count
    assert (jc[0] == 2).all() and jc.min() <= 1 and jc.max() >= 3
    assert outs["done"].sum() >= 2 * 6 * W                 # >= 2 episode ends per world
    # entity generations advance when the 27 bodies are recreated
    assert outs["body_entity"][-1][:, 0].max() >= 2
    # hiders held something at some point (fixed joint), seekers shoved (hinge)
    holding = outs["self_obs"][..., 8]
    assert (holding == 1).any() and (holding == 2).any()
    # doors stay put while latched (first steps), line-of-sight flags vary
    door0 = np.stack([f[15] for f in pos[:5]])
    assert np.abs(door0[:, :2] - door0[0, :2]).max() < 1e-3
    vis = outs["other_obs"][..., 3]
    assert 0.02 < vis.mean() < 0.98
    # tilted bodies exist (ramps / shoved boxes): rotations are not yaw-only
    rot = np.concatenate(outs["body_rot"])
    assert (np.abs(rot[:, 1]) + np.abs(rot[:, 2]) > 0.05).any()


@pytest.mark.gpu
def test_gpu_matches_golden():
    W, steps, ins, outs = load_golden("arena_w2_s200")
    got, n_kernels = rollout_gpu("arena", W, steps, ins, CFG)
    assert n_kernels > 10
    assert_traces_equal(got, outs, exact=EXACT, rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_independent_nodes_become_graph_branches(monkeypatch):
    # selfObs / otherObs / lidar only depend on the post-reset broadphase update
    # (sims/arena/sim.cpp setupTasks): the step graph must fork, and forking must not
    # change a bit of the result
    from sims import make_executor
    W, steps, ins, outs = load_golden("arena_w2_s200")
    ex = make_executor("arena", W, **CFG)
    g = ex.buildLaunchGraphAllTaskGraphs()
    assert g.num_branches >= 3
    del g
    ex.close()
    monkeypatch.setenv("MADRONA_B200_GRAPH_BRANCHES", "0")
    ex = make_executor("arena", W, **CFG)
    g = ex.buildLaunchGraphAllTaskGraphs()
    assert g.num_branches == 1
    del g
    ex.close()
    short = {k: v[:40] for k, v in ins.items()}
    got, _ = rollout_gpu("arena", W, 40, short, CFG)
    assert_traces_equal(got, {k: v[:41] for k, v in outs.items()}, exact=EXACT, rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_gpu_matches_live_reference_many_worlds():
    # the reference CPU backend's trace is stored as a digest golden (tests/golden/make_golden.py)
    W, steps = 160, 150
    cfg = {"episode_len": 60, "seed": 4000}
    ins = make_inputs("arena", W, steps, seed=21)
    got, _ = rollout_gpu("arena", W, steps, ins, cfg)
    assert_matches_digest_golden(got, "arena_w160_s150_ref", ins, exact=EXACT, rtol=1e-4, atol=1e-5)
